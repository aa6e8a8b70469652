/*
 * bench_cigar_inputs.c -- cigars in on the flat C-ABI by two routes, for tools/bench_cigar_inputs.py.  Every pair is a LEN-base sequence X
 * and a copy Y evolved from it (8 % substitutions, 1 % insertions and 1 % deletions of 1-3 bases), with the cigar of that evolution;
 * cPecanRealign's parameters (trim 0, expansion 4, split 10), five-state default model.  Per batch of BATCH pairs:
 *   anchors, host route: convertPairwiseForwardStrandAlignmentToAnchorPairs + columns_match on THREADS threads, then cpb_batch_create;
 *   anchors, device route: cpb_batch_create_from_cigars;
 *   rescoring, host route: after an ALIGNED_PAIRS run, cpb_batch_fetch_pairs_reference_order of list 0, then on THREADS threads every pair's
 *     columns weighed against it (score_anchor_pairs), scoreByPosteriorProbability and the cigar of the columns (pairs_to_alignment);
 *   rescoring, device route: after the same run, cpb_batch_alignments_from_cigars, cpb_batch_score_alignments(CPB_SCORE_POSTERIOR),
 *     cpb_batch_alignment_cigars and cpb_batch_fetch_cigars.
 * Each time is the sum over the batches of one repetition; REPS repetitions follow a warm-up.  Every pair's anchors, score bits and cigar
 * are compared between the routes.  One JSON line on stdout.
 *
 *   bench_cigar_inputs NPAIRS LEN BATCH THREADS REPS
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

static void check(int rc, const char *what) {
    if (rc != CPB_OK) {
        fprintf(stderr, "bench_cigar_inputs: %s: %s\n", what, cpb_last_error());
        exit(1);
    }
}

static void *xmalloc(size_t bytes) {
    void *p = malloc(bytes ? bytes : 1);
    if (p == NULL) {
        fprintf(stderr, "bench_cigar_inputs: out of memory\n");
        exit(2);
    }
    return p;
}

static int cmp_double(const void *a, const void *b) {
    const double x = *(const double *) a, y = *(const double *) b;
    return x < y ? -1 : (x > y ? 1 : 0);
}

/* {"median":, "min":, "max":} of n values */
static void stat_json(char *out, const char *name, double *v, int n) {
    qsort(v, (size_t) n, sizeof(double), cmp_double);
    sprintf(out + strlen(out), "\"%s\": {\"median\": %.6f, \"min\": %.6f, \"max\": %.6f}, ", name, v[n / 2], v[0], v[n - 1]);
}

static uint64_t rng_state = 88172645463325252ULL;
static uint64_t rnd(void) {
    rng_state ^= rng_state << 13;
    rng_state ^= rng_state >> 7;
    rng_state ^= rng_state << 17;
    return rng_state;
}
static double unif(void) { return (double) (rnd() >> 11) * (1.0 / 9007199254740992.0); }

/* one batch: sequences, offsets, cigars */
typedef struct {
    int64_t n, *xOff, *yOff, *opOff;
    char *seqX, *seqY;
    int32_t *ops;
} Inputs;

static void add_op(int32_t *ops, int64_t *m, int32_t type, int32_t len) {
    if (*m > 0 && ops[2 * (*m - 1)] == type) ops[2 * (*m - 1) + 1] += len;
    else {
        ops[2 * *m] = type;
        ops[2 * *m + 1] = len;
        (*m)++;
    }
}

static int base_index(char c) { return c == 'A' ? 0 : (c == 'C' ? 1 : (c == 'G' ? 2 : 3)); }

static void make_inputs(Inputs *in, int64_t n, int64_t len) {
    static const char acgt[4] = { 'A', 'C', 'G', 'T' };
    in->n = n;
    in->xOff = xmalloc((size_t) (n + 1) * 8);
    in->yOff = xmalloc((size_t) (n + 1) * 8);
    in->opOff = xmalloc((size_t) (n + 1) * 8);
    in->seqX = xmalloc((size_t) (n * len));
    in->seqY = xmalloc((size_t) (n * len * 2));
    in->ops = xmalloc((size_t) (n * len * 2 + 16) * 2 * sizeof(int32_t));
    int64_t x = 0, y = 0, m = 0;
    in->xOff[0] = in->yOff[0] = in->opOff[0] = 0;
    for (int64_t i = 0; i < n; i++) {
        const int64_t x0 = x;
        for (int64_t k = 0; k < len; k++) in->seqX[x++] = acgt[rnd() & 3];
        int32_t *ops = in->ops + 2 * m;
        int64_t mi = 0;
        for (int64_t k = x0; k < x; k++) {
            const double r = unif();
            if (r < 0.01) { /* insertion in Y before this base */
                const int32_t l = 1 + (int32_t) (rnd() % 3);
                for (int32_t j = 0; j < l; j++) in->seqY[y++] = acgt[rnd() & 3];
                add_op(ops, &mi, CPB_OP_INDEL_Y, l);
            } else if (r < 0.02) { /* deletion of this base and up to two more */
                int32_t l = 1 + (int32_t) (rnd() % 3);
                if (k + l > x) l = (int32_t) (x - k);
                add_op(ops, &mi, CPB_OP_INDEL_X, l);
                k += l - 1;
                continue;
            }
            in->seqY[y++] = unif() < 0.08 ? acgt[(base_index(in->seqX[k]) + 1 + (int) (rnd() % 3)) & 3] : in->seqX[k];
            add_op(ops, &mi, CPB_OP_MATCH, 1);
        }
        m += mi;
        in->xOff[i + 1] = x;
        in->yOff[i + 1] = y;
        in->opOff[i + 1] = m;
    }
}

/* ---- host routes, pairs dealt to threads ---- */
typedef struct {
    const Inputs *in;
    int64_t trim, expansion;
    /* anchors: per pair an int64 (x, y, e) array */
    int64_t **anchors, *nAnchors;
    /* rescoring: list 0 in reference order, the score and the cigar of every pair */
    const int64_t *l0Off;
    const int32_t *l0;
    double *score;
    int32_t **cig;
    int64_t *nCig;
    int64_t next;
    pthread_mutex_t lock;
} Work;

static int64_t take(Work *w) {
    pthread_mutex_lock(&w->lock);
    const int64_t i = w->next < w->in->n ? w->next++ : -1;
    pthread_mutex_unlock(&w->lock);
    return i;
}

/* convertPairwiseForwardStrandAlignmentToAnchorPairs of pair i's cigar: every column, unfiltered */
static stList *cigar_columns(const Work *w, int64_t i) {
    const Inputs *in = w->in;
    struct List *ops = constructEmptyList(0, (void (*)(void *)) destructAlignmentOperation);
    for (int64_t k = in->opOff[i]; k < in->opOff[i + 1]; k++) listAppend(ops, constructAlignmentOperation(in->ops[2 * k], in->ops[2 * k + 1], 0.0));
    struct PairwiseAlignment *pA = constructPairwiseAlignment("x", 0, in->xOff[i + 1] - in->xOff[i], 1, "y", 0, in->yOff[i + 1] - in->yOff[i], 1, 0.0, ops);
    stList *cols = convertPairwiseForwardStrandAlignmentToAnchorPairs(pA, w->trim, w->expansion);
    destructPairwiseAlignment(pA);
    return cols;
}

static void *anchors_thread(void *arg) {
    Work *w = arg;
    const Inputs *in = w->in;
    for (int64_t i; (i = take(w)) >= 0;) {
        stList *cols = cigar_columns(w, i);
        const char *sX = in->seqX + in->xOff[i], *sY = in->seqY + in->yOff[i];
        const int64_t n = stList_length(cols);
        int64_t *a = xmalloc((size_t) (n > 0 ? n : 1) * 3 * sizeof(int64_t)), k = 0;
        for (int64_t j = 0; j < n; j++) {
            stIntTuple *t = stList_get(cols, j);
            const int64_t x = stIntTuple_get(t, 0), y = stIntTuple_get(t, 1);
            const int cx = toupper((unsigned char) sX[x]), cy = toupper((unsigned char) sY[y]);
            if (cx == cy && cx != 'N') { /* columns_match */
                a[3 * k] = x;
                a[3 * k + 1] = y;
                a[3 * k + 2] = stIntTuple_get(t, 2);
                k++;
            }
        }
        stList_destruct(cols);
        w->anchors[i] = a;
        w->nAnchors[i] = k;
    }
    return NULL;
}

static int by_xy(const void *a, const void *b) {
    const int64_t *p = a, *q = b;
    if (p[0] != q[0]) return p[0] < q[0] ? -1 : 1;
    return p[1] < q[1] ? -1 : (p[1] > q[1] ? 1 : 0);
}

static void *rescore_thread(void *arg) {
    Work *w = arg;
    const Inputs *in = w->in;
    for (int64_t i; (i = take(w)) >= 0;) {
        stList *cols = cigar_columns(w, i);
        const int64_t n = stList_length(cols), lX = in->xOff[i + 1] - in->xOff[i], lY = in->yOff[i + 1] - in->yOff[i];
        int64_t *a = xmalloc((size_t) (n > 0 ? n : 1) * 3 * sizeof(int64_t)); /* (x, y, weight or -1): score_anchor_pairs */
        for (int64_t j = 0; j < n; j++) {
            stIntTuple *t = stList_get(cols, j);
            a[3 * j] = stIntTuple_get(t, 0);
            a[3 * j + 1] = stIntTuple_get(t, 1);
            a[3 * j + 2] = -1;
        }
        stList_destruct(cols);
        qsort(a, (size_t) n, 3 * sizeof(int64_t), by_xy);
        int32_t *scored = xmalloc((size_t) (n > 0 ? n : 1) * 3 * sizeof(int32_t));
        int64_t s = 0;
        for (int64_t k = w->l0Off[i]; k < w->l0Off[i + 1]; k++) {
            int64_t key[3] = { w->l0[3 * k + 1], w->l0[3 * k + 2], 0 };
            int64_t *hit = bsearch(key, a, (size_t) n, 3 * sizeof(int64_t), by_xy);
            if (hit != NULL && hit[2] < 0) {
                hit[2] = w->l0[3 * k];
                scored[3 * s] = (int32_t) hit[2];
                scored[3 * s + 1] = (int32_t) hit[0];
                scored[3 * s + 2] = (int32_t) hit[1];
                s++;
            }
        }
        for (int64_t j = 0; j < n; j++) {
            if (a[3 * j + 2] < 0) {
                scored[3 * s] = 0;
                scored[3 * s + 1] = (int32_t) a[3 * j];
                scored[3 * s + 2] = (int32_t) a[3 * j + 1];
                s++;
            }
        }
        stList *l = cpecan_tripleList_construct(scored, s);
        w->score[i] = scoreByPosteriorProbability(lX, lY, l);
        stList_destruct(l);
        free(scored);
        /* the cigar of the columns, which a holds in (x, y) order: pairs_to_alignment */
        int32_t *c = xmalloc((size_t) (3 * n + 2) * 2 * sizeof(int32_t));
        int64_t m = 0, px = -1, py = -1;
        for (int64_t j = 0; j <= n; j++) {
            const int64_t x = j < n ? a[3 * j] : lX, y = j < n ? a[3 * j + 1] : lY;
            if (x - px > 1) add_op(c, &m, CPB_OP_INDEL_X, (int32_t) (x - px - 1));
            if (y - py > 1) add_op(c, &m, CPB_OP_INDEL_Y, (int32_t) (y - py - 1));
            if (j < n) add_op(c, &m, CPB_OP_MATCH, 1);
            px = x;
            py = y;
        }
        free(a);
        w->cig[i] = c;
        w->nCig[i] = m;
    }
    return NULL;
}

static void run_threads(Work *w, int threads, void *(*fn)(void *)) {
    pthread_t *t = xmalloc((size_t) threads * sizeof(pthread_t));
    w->next = 0;
    for (int k = 0; k < threads; k++) pthread_create(&t[k], NULL, fn, w);
    for (int k = 0; k < threads; k++) pthread_join(t[k], NULL);
    free(t);
}

int main(int argc, char **argv) {
    if (argc != 6) {
        fprintf(stderr, "usage: bench_cigar_inputs NPAIRS LEN BATCH THREADS REPS\n");
        return 2;
    }
    const int64_t nAll = atoll(argv[1]), len = atoll(argv[2]), batch = atoll(argv[3]);
    const int threads = atoi(argv[4]), reps = atoi(argv[5]);
    const int nb = (int) ((nAll + batch - 1) / batch);
    CpbParams p;
    cpb_params_default(&p);
    p.constraintDiagonalTrim = 0;
    p.diagonalExpansion = 4;
    p.splitMatrixBiggerThanThis = 10;
    CpbModel model;
    check(cpb_model_default(CPB_FIVE_STATE, &model), "model");
    cpb_context *ctx;
    check(cpb_context_create(0, NULL, &ctx), "context");
    Inputs *in = xmalloc((size_t) nb * sizeof(Inputs));
    for (int k = 0; k < nb; k++) make_inputs(&in[k], k + 1 < nb ? batch : nAll - (int64_t) k * batch, len);
    double *tHostA = xmalloc(sizeof(double) * reps), *tDevA = xmalloc(sizeof(double) * reps), *tRun = xmalloc(sizeof(double) * reps),
           *tHostR = xmalloc(sizeof(double) * reps), *tDevR = xmalloc(sizeof(double) * reps);
    int64_t differ = 0, pairs = 0, nOpsAll = 0, nAnchorsAll = 0, nList0 = 0, nColsAll = 0, nCigOps = 0;
    for (int rep = -1; rep < reps; rep++) { /* rep -1: the warm-up */
        double hA = 0, dA = 0, run = 0, hR = 0, dR = 0;
        for (int k = 0; k < nb; k++) {
            const Inputs *I = &in[k];
            const int64_t n = I->n;
            Work w;
            memset(&w, 0, sizeof(w));
            pthread_mutex_init(&w.lock, NULL);
            w.in = I;
            w.trim = p.constraintDiagonalTrim;
            w.expansion = p.diagonalExpansion;
            /* anchors */
            double t0 = now();
            w.anchors = xmalloc((size_t) n * sizeof(int64_t *));
            w.nAnchors = xmalloc((size_t) n * sizeof(int64_t));
            run_threads(&w, threads, anchors_thread);
            int64_t *aOff = xmalloc((size_t) (n + 1) * 8);
            aOff[0] = 0;
            for (int64_t i = 0; i < n; i++) aOff[i + 1] = aOff[i] + w.nAnchors[i];
            int64_t *flat = xmalloc((size_t) (aOff[n] > 0 ? aOff[n] : 1) * 3 * 8);
            for (int64_t i = 0; i < n; i++) {
                memcpy(flat + 3 * aOff[i], w.anchors[i], (size_t) w.nAnchors[i] * 3 * 8);
                free(w.anchors[i]);
            }
            cpb_batch *hb, *db;
            check(cpb_batch_create(ctx, n, I->seqX, I->xOff, I->seqY, I->yOff, flat, aOff, NULL, NULL, &hb), "cpb_batch_create");
            hA += now() - t0;
            t0 = now();
            check(cpb_batch_create_from_cigars(ctx, n, I->seqX, I->xOff, I->seqY, I->yOff, I->opOff, I->ops, NULL, NULL, &p, &db), "cpb_batch_create_from_cigars");
            dA += now() - t0;
            if (rep == reps - 1) { /* compare the anchors once */
                const int64_t m = cpb_batch_anchor_count(db);
                int64_t *o2 = xmalloc((size_t) (n + 1) * 8), *t2 = xmalloc((size_t) (m > 0 ? m : 1) * 3 * 8);
                check(cpb_batch_fetch_anchors(db, o2, t2), "fetch anchors");
                for (int64_t i = 0; i < n; i++) {
                    if (o2[i + 1] - o2[i] != aOff[i + 1] - aOff[i] || memcmp(t2 + 3 * o2[i], flat + 3 * aOff[i], (size_t) (aOff[i + 1] - aOff[i]) * 24) != 0) differ++;
                }
                free(o2);
                free(t2);
                nAnchorsAll += aOff[n];
                nOpsAll += I->opOff[n];
                pairs += n;
            }
            free(flat);
            free(aOff);
            free(w.anchors);
            free(w.nAnchors);
            cpb_batch_destroy(hb);
            /* rescoring */
            t0 = now();
            check(cpb_batch_run(db, &model, &p, CPB_MODE_ALIGNED_PAIRS), "run");
            run += now() - t0;
            t0 = now();
            const int64_t m0 = cpb_batch_result_count(db, 0);
            int64_t *l0Off = xmalloc((size_t) (n + 1) * 8);
            int32_t *l0 = xmalloc((size_t) (m0 > 0 ? m0 : 1) * 12);
            check(cpb_batch_fetch_pairs_reference_order(db, 0, l0Off, l0), "fetch list 0");
            w.l0Off = l0Off;
            w.l0 = l0;
            w.score = xmalloc((size_t) n * sizeof(double));
            w.cig = xmalloc((size_t) n * sizeof(int32_t *));
            w.nCig = xmalloc((size_t) n * sizeof(int64_t));
            run_threads(&w, threads, rescore_thread);
            hR += now() - t0;
            t0 = now();
            double *score = xmalloc((size_t) n * sizeof(double));
            int64_t *cOff = xmalloc((size_t) (n + 1) * 8);
            check(cpb_batch_alignments_from_cigars(db, I->opOff, I->ops, p.constraintDiagonalTrim), "cpb_batch_alignments_from_cigars");
            check(cpb_batch_score_alignments(db, CPB_SCORE_POSTERIOR, score), "score");
            check(cpb_batch_alignment_cigars(db, cOff), "cigars");
            int32_t *cig = xmalloc((size_t) (cOff[n] > 0 ? cOff[n] : 1) * 8);
            check(cpb_batch_fetch_cigars(db, cig), "fetch cigars");
            dR += now() - t0;
            if (rep == reps - 1) {
                for (int64_t i = 0; i < n; i++) {
                    if (memcmp(&score[i], &w.score[i], sizeof(double)) != 0 || cOff[i + 1] - cOff[i] != w.nCig[i] ||
                        memcmp(cig + 2 * cOff[i], w.cig[i], (size_t) w.nCig[i] * 8) != 0)
                        differ++;
                }
                nList0 += m0;
                nColsAll += cpb_batch_alignments_count(db);
                nCigOps += cOff[n];
            }
            for (int64_t i = 0; i < n; i++) free(w.cig[i]);
            free(w.cig);
            free(w.nCig);
            free(w.score);
            free(score);
            free(cOff);
            free(cig);
            free(l0);
            free(l0Off);
            cpb_batch_destroy(db);
        }
        if (rep >= 0) {
            tHostA[rep] = hA;
            tDevA[rep] = dA;
            tRun[rep] = run;
            tHostR[rep] = hR;
            tDevR[rep] = dR;
        }
    }
    /* bytes across the link, from the counts and the copies each entry point makes: the sequences, common to both routes, are left out; the
     * device rescoring uploads the offsets of the cigars, the columns, list 0 and both sequences, and again two tables each for the score and
     * the cigar build */
    const int64_t offs = (nAll + nb) * 8;
    char out[4096] = "{";
    sprintf(out + strlen(out), "\"pairs\": %" PRId64 ", \"batches\": %d, \"operations\": %" PRId64 ", \"anchors\": %" PRId64 ", \"list0_triples\": %" PRId64
                               ", \"columns\": %" PRId64 ", \"cigar_operations\": %" PRId64 ", ",
            pairs, nb, nOpsAll, nAnchorsAll, nList0, nColsAll, nCigOps);
    stat_json(out, "s_anchors_host", tHostA, reps);
    stat_json(out, "s_anchors_device", tDevA, reps);
    stat_json(out, "s_run", tRun, reps);
    stat_json(out, "s_rescore_host", tHostR, reps);
    stat_json(out, "s_rescore_device", tDevR, reps);
    sprintf(out + strlen(out),
            "\"bytes\": {\"anchors_host_h2d\": %" PRId64 ", \"anchors_host_d2h\": 0, \"anchors_device_h2d\": %" PRId64 ", \"anchors_device_d2h\": %" PRId64
            ", \"rescore_host_h2d\": 0, \"rescore_host_d2h\": %" PRId64 ", \"rescore_device_h2d\": %" PRId64 ", \"rescore_device_d2h\": %" PRId64 "}, ",
            12 * nAnchorsAll + 3 * offs, 8 * nOpsAll + 3 * offs, 12 * nAnchorsAll + offs, 12 * nList0 + offs, 8 * nOpsAll + 11 * offs,
            8 * nCigOps + 8 * nAll + offs);
    sprintf(out + strlen(out), "\"pairs_differing\": %" PRId64 "}", differ);
    puts(out);
    cpb_context_destroy(ctx);
    return differ != 0;
}
