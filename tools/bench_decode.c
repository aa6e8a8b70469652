/*
 * bench_decode.c -- the device decoders of the flat C-ABI (cpb_batch_ordered_chain, cpb_batch_mea) against libcpecan.so's host functions
 * (host/realign.c) on the same lists, for tools/bench_device_alignments.py.  The batch is anchored on the device and run once; then
 *   chain: device reweight + chain vs host reweightAlignedPairs2 + filterPairwiseAlignmentToMakePairsOrdered over the fetched list 0
 *          (reweight < 0: no reweighting, the chain alone);
 *   mea:   device MEA + left shift vs host getMaximalExpectedAccuracyPairwiseAlignment + leftShiftAlignment over the lists in the
 *          reference's order (cpb_batch_fetch_pairs_reference_order, what libcpecan.so hands over).
 * Device time: median of REPS synchronised calls after a warm-up (the chain's batch is run again before each, not timed).  Host time: the
 * functions alone on THREADS threads, their input lists built beforehand.  Every pair is compared.  One JSON line on stdout.
 *
 *   bench_decode SEQS.bin chain|mea TRIM EXPANSION SPLIT GAMMA REWEIGHT THREADS REPS
 *   SEQS.bin: int64 n; int64 xOff[n+1], yOff[n+1]; char seqX[xOff[n]], seqY[yOff[n]]
 */
#include <inttypes.h>
#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "cpecan/multipleAligner.h"
#include "cpecan/pairwiseAligner.h"
#include "cpecan_b200.h"

stList *cpecan_tripleList_construct(const int32_t *triples, int64_t n); /* host/containers.c: a list whose tuples come from one slab */

static double now(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double) ts.tv_sec + 1e-9 * (double) ts.tv_nsec;
}

static void *read_block(FILE *f, size_t bytes) {
    void *p = malloc(bytes ? bytes : 1);
    if (p == NULL || fread(p, 1, bytes, f) != bytes) {
        fprintf(stderr, "bench_decode: short read\n");
        exit(2);
    }
    return p;
}

static void check(int rc, const char *what) {
    if (rc != CPB_OK) {
        fprintf(stderr, "bench_decode: %s: %s\n", what, cpb_last_error());
        exit(1);
    }
}

static int cmp_double(const void *a, const void *b) {
    const double x = *(const double *) a, y = *(const double *) b;
    return x < y ? -1 : (x > y ? 1 : 0);
}

typedef struct {
    int64_t n, *xOff, *yOff;
    char **sX, **sY;
    stList **in0, **in1, **in2, **out;
    double *score;
    int mea;
    float gamma;
    double reweight;
    int64_t next, stride;
    pthread_mutex_t lock;
} Work;

static void *host_worker(void *arg) {
    Work *w = arg;
    PairwiseAlignmentParameters *p = pairwiseAlignmentBandingParameters_construct();
    p->gapGamma = w->gamma;
    for (;;) {
        pthread_mutex_lock(&w->lock);
        const int64_t i0 = w->next;
        w->next += w->stride;
        pthread_mutex_unlock(&w->lock);
        if (i0 >= w->n) break;
        const int64_t i1 = i0 + w->stride < w->n ? i0 + w->stride : w->n;
        for (int64_t i = i0; i < i1; i++) {
            const int64_t lX = w->xOff[i + 1] - w->xOff[i], lY = w->yOff[i + 1] - w->yOff[i];
            if (w->mea) {
                stList *m = getMaximalExpectedAccuracyPairwiseAlignment(w->in0[i], w->in1[i], w->in2[i], lX, lY, &w->score[i], p);
                w->out[i] = leftShiftAlignment(m, w->sX[i], w->sY[i]);
                stList_destruct(m);
            } else {
                stList *l = w->reweight >= 0 ? reweightAlignedPairs2(w->in0[i], lX, lY, w->reweight) : w->in0[i];
                w->out[i] = filterPairwiseAlignmentToMakePairsOrdered(l, w->sX[i], w->sY[i], w->gamma);
                w->in0[i] = NULL; /* consumed */
            }
        }
    }
    pairwiseAlignmentBandingParameters_destruct(p);
    return NULL;
}

static stList **lists_of(int64_t n, const int64_t *off, const int32_t *tri) {
    stList **l = malloc((size_t) (n > 0 ? n : 1) * sizeof(stList *));
    for (int64_t i = 0; i < n; i++) l[i] = cpecan_tripleList_construct(tri + 3 * off[i], off[i + 1] - off[i]);
    return l;
}

int main(int argc, char **argv) {
    if (argc < 10) {
        fprintf(stderr, "usage: %s SEQS.bin chain|mea TRIM EXPANSION SPLIT GAMMA REWEIGHT THREADS REPS\n", argv[0]);
        return 2;
    }
    FILE *f = fopen(argv[1], "rb");
    if (f == NULL) {
        perror(argv[1]);
        return 2;
    }
    const int mea = strcmp(argv[2], "mea") == 0;
    int64_t n;
    if (fread(&n, sizeof(n), 1, f) != 1) return 2;
    int64_t *xOff = read_block(f, (size_t) (n + 1) * 8), *yOff = read_block(f, (size_t) (n + 1) * 8);
    char *seqX = read_block(f, (size_t) xOff[n]), *seqY = read_block(f, (size_t) yOff[n]);
    fclose(f);
    CpbParams cp;
    cpb_params_default(&cp);
    cp.constraintDiagonalTrim = atoll(argv[3]);
    cp.diagonalExpansion = atoll(argv[4]);
    cp.splitMatrixBiggerThanThis = atoll(argv[5]);
    const float gamma = (float) atof(argv[6]);
    const double reweight = atof(argv[7]);
    const int threads = atoi(argv[8]), reps = atoi(argv[9]);

    cpb_context *ctx;
    cpb_batch *b;
    CpbModel m;
    check(cpb_context_create(0, NULL, &ctx), "context");
    check(cpb_model_default(CPB_FIVE_STATE, &m), "model");
    check(cpb_batch_create_anchored(ctx, n, seqX, xOff, seqY, yOff, NULL, NULL, &cp, &b), "create");
    const int mode = mea ? CPB_MODE_ALIGNED_PAIRS_INDELS : CPB_MODE_ALIGNED_PAIRS;
    check(cpb_batch_run(b, &m, &cp, mode), "run");
    fprintf(stderr, "bench_decode: %" PRIi64 " pairs anchored and run\n", n);

    /* the host arm's inputs: the lists as libcpecan.so hands them over */
    const int nLists = mea ? 3 : 1;
    int64_t *off[3] = { NULL, NULL, NULL }, cloud = 0;
    int32_t *tri[3] = { NULL, NULL, NULL };
    for (int l = 0; l < nLists; l++) {
        const int64_t c = cpb_batch_result_count(b, l);
        cloud += c;
        off[l] = malloc((size_t) (n + 1) * 8);
        tri[l] = malloc((size_t) (c > 0 ? c : 1) * 12);
        check(mea ? cpb_batch_fetch_pairs_reference_order(b, l, off[l], tri[l]) : cpb_batch_fetch_pairs(b, l, off[l], tri[l]), "fetch");
    }
    Work w;
    memset(&w, 0, sizeof(w));
    w.n = n;
    w.xOff = xOff;
    w.yOff = yOff;
    w.sX = malloc((size_t) (n > 0 ? n : 1) * sizeof(char *));
    w.sY = malloc((size_t) (n > 0 ? n : 1) * sizeof(char *));
    for (int64_t i = 0; i < n; i++) {
        const int64_t lX = xOff[i + 1] - xOff[i], lY = yOff[i + 1] - yOff[i];
        w.sX[i] = malloc((size_t) lX + 1);
        w.sY[i] = malloc((size_t) lY + 1);
        memcpy(w.sX[i], seqX + xOff[i], (size_t) lX);
        memcpy(w.sY[i], seqY + yOff[i], (size_t) lY);
        w.sX[i][lX] = w.sY[i][lY] = 0;
    }
    w.in0 = lists_of(n, off[0], tri[0]);
    if (mea) {
        w.in1 = lists_of(n, off[1], tri[1]);
        w.in2 = lists_of(n, off[2], tri[2]);
    }
    w.out = calloc((size_t) (n > 0 ? n : 1), sizeof(stList *));
    w.score = calloc((size_t) (n > 0 ? n : 1), sizeof(double));
    w.mea = mea;
    w.gamma = gamma;
    w.reweight = reweight;
    w.stride = 64;
    pthread_mutex_init(&w.lock, NULL);
    pthread_t *th = malloc((size_t) threads * sizeof(pthread_t));
    double t0 = now();
    for (int t = 0; t < threads; t++) pthread_create(&th[t], NULL, host_worker, &w);
    for (int t = 0; t < threads; t++) pthread_join(th[t], NULL);
    const double hostMs = 1e3 * (now() - t0);
    fprintf(stderr, "bench_decode: host arm %.1f ms\n", hostMs);

    /* the device arm: a warm-up, then REPS timed calls */
    double *dev = malloc((size_t) (reps + 1) * sizeof(double)), *scores = malloc((size_t) (n > 0 ? n : 1) * sizeof(double));
    for (int r = 0; r <= reps; r++) {
        if (!mea && r > 0) check(cpb_batch_run(b, &m, &cp, mode), "run");
        t0 = now();
        if (mea) {
            check(cpb_batch_mea(b, gamma, 1, scores), "mea");
        } else {
            if (reweight >= 0) check(cpb_batch_reweight_pairs(b, reweight), "reweight");
            check(cpb_batch_ordered_chain(b, gamma), "chain");
        }
        dev[r] = 1e3 * (now() - t0);
    }
    qsort(dev + 1, (size_t) reps, sizeof(double), cmp_double);
    const int64_t alnCount = cpb_batch_alignments_count(b);
    int64_t *aOff = malloc((size_t) (n + 1) * 8);
    int32_t *aTri = malloc((size_t) (alnCount > 0 ? alnCount : 1) * 12);
    check(cpb_batch_fetch_alignments(b, aOff, aTri), "fetch alignments");

    int64_t differ = 0, first = -1;
    for (int64_t i = 0; i < n; i++) {
        stList *o = w.out[i];
        const int64_t len = stList_length(o);
        int same = len == aOff[i + 1] - aOff[i];
        for (int64_t k = 0; same && k < len; k++) {
            stIntTuple *t = stList_get(o, k);
            const int32_t *d = aTri + 3 * (aOff[i] + k);
            same = stIntTuple_get(t, 0) == d[0] && stIntTuple_get(t, 1) == d[1] && stIntTuple_get(t, 2) == d[2];
        }
        if (mea) same = same && memcmp(&w.score[i], &scores[i], sizeof(double)) == 0;
        if (!same) {
            differ++;
            if (first < 0) first = i;
        }
    }
    printf("{\"pairs\": %" PRIi64 ", \"cloud_triples\": %" PRIi64 ", \"cloud_bytes\": %" PRIi64 ", \"alignment_triples\": %" PRIi64
           ", \"alignment_bytes\": %" PRIi64 ", \"host_threads\": %d, \"host_ms\": %.1f, \"device_ms\": %.2f, \"device_ms_all\": [",
           n, cloud, cloud * 12 + (int64_t) nLists * (n + 1) * 8, alnCount, alnCount * 12 + (n + 1) * 8, threads, hostMs, dev[1 + reps / 2]);
    for (int r = 1; r <= reps; r++) printf("%s%.2f", r > 1 ? ", " : "", dev[r]);
    printf("], \"warmup_ms\": %.2f, \"pairs_checked\": %" PRIi64 ", \"pairs_differing\": %" PRIi64 ", \"first_differing\": %" PRIi64 "}\n", dev[0], n,
           differ, first);
    cpb_batch_destroy(b);
    cpb_context_destroy(ctx);
    return differ != 0;
}
