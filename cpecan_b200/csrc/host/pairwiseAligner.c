/*
 * host/pairwiseAligner.c -- cPecan's pairwise-alignment entry points (inc/pairwiseAligner.h of the reference) as
 * plain C over the batched CUDA engine (include/cpecan_b200.h).
 *
 * What the reference does per call on the host -- split at large anchor gaps, build the band, run the banded
 * forward / backward sweeps block by block, threshold the posteriors (impl/pairwiseAligner.c:756-877, :1273-1326,
 * :1431-1513) -- happens on the device inside cpb_batch_run.  This file only translates between the reference's
 * argument conventions (NUL-terminated strings, stList of stIntTuple) and the engine's flat batch, for one pair
 * (the reference's own signatures) or many (the *Batch forms).  There is no host implementation of the DP here.
 */
#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

#include "cpecan/pairwiseAligner.h"
#include "cpecan_b200.h"
#include "host_internal.h"
#include "minijson.h"

const char *PAIRWISE_ALIGNMENT_EXCEPTION_ID = "PAIRWISE_ALIGNMENT_EXCEPTION";

void *cpecan_malloc(size_t bytes) {
    void *p = malloc(bytes ? bytes : 1);
    if (p == NULL) st_errAbort("cpecan: out of memory allocating %zu bytes", bytes);
    return p;
}

static double wall_seconds(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double) ts.tv_sec + 1e-9 * (double) ts.tv_nsec;
}

/* ------------------------------------------------------------------------- host threads for the marshalling */

/* The reference's interface hands every aligned pair over as a heap tuple in a list: for a batch of 100 000 x 1 kb pairs that is 1e8
 * tuples in and out of the call, which a single thread needs seconds for while the device pass takes one.  Problems are independent,
 * so the conversions run on a few host threads over contiguous ranges of problems. */
typedef struct {
    void (*fn)(int64_t, int64_t, void *);
    void *arg;
    int64_t first, last;
} ParallelTask;

static void *parallel_entry(void *v) {
    ParallelTask *t = v;
    t->fn(t->first, t->last, t->arg);
    return NULL;
}

void cpecan_parallel_for(int64_t n, const int64_t *weight, void (*fn)(int64_t first, int64_t last, void *arg), void *arg) {
    long threads = sysconf(_SC_NPROCESSORS_ONLN);
    const char *e = getenv("CPECAN_HOST_THREADS");
    if (e != NULL) threads = atol(e);
    if (threads > 32) threads = 32;
    const int64_t total = weight != NULL ? weight[n] - weight[0] : n;
    if (threads > n) threads = (long) n;
    if (threads <= 1 || total < 200000) { /* not worth a thread */
        if (n > 0) fn(0, n, arg);
        return;
    }
    ParallelTask tasks[32];
    pthread_t ids[32];
    int64_t at = 0;
    int started = 0;
    for (long t = 0; t < threads; t++) {
        int64_t end = n;
        if (t + 1 < threads) {
            if (weight == NULL) {
                end = n * (t + 1) / threads;
            } else { /* first index whose prefix weight reaches this thread's share */
                const int64_t want = weight[0] + total * (t + 1) / threads;
                int64_t lo = at, hi = n;
                while (lo < hi) {
                    const int64_t mid = lo + (hi - lo) / 2;
                    if (weight[mid] < want) lo = mid + 1;
                    else hi = mid;
                }
                end = lo;
            }
        }
        if (end <= at) continue;
        tasks[started].fn = fn;
        tasks[started].arg = arg;
        tasks[started].first = at;
        tasks[started].last = end;
        if (pthread_create(&ids[started], NULL, parallel_entry, &tasks[started]) != 0) { /* no thread: do the range here */
            fn(at, end, arg);
        } else {
            started++;
        }
        at = end;
    }
    for (int t = 0; t < started; t++) pthread_join(ids[t], NULL);
}

/* ------------------------------------------------------------------------------------ parameters */

PairwiseAlignmentParameters *pairwiseAlignmentBandingParameters_construct(void) {
    /* one source of truth for the defaults of impl/pairwiseAligner.c:1334-1348: the engine's cpb_params_default */
    CpbParams d;
    cpb_params_default(&d);
    PairwiseAlignmentParameters *p = cpecan_malloc(sizeof(*p));
    p->threshold = d.threshold;
    p->minDiagsBetweenTraceBack = d.minDiagsBetweenTraceBack;
    p->traceBackDiagonals = d.traceBackDiagonals;
    p->diagonalExpansion = d.diagonalExpansion;
    p->constraintDiagonalTrim = d.constraintDiagonalTrim;
    p->anchorMatrixBiggerThanThis = d.anchorMatrixBiggerThanThis;
    p->repeatMaskMatrixBiggerThanThis = d.repeatMaskMatrixBiggerThanThis;
    p->splitMatrixBiggerThanThis = d.splitMatrixBiggerThanThis;
    p->alignAmbiguityCharacters = d.alignAmbiguityCharacters != 0;
    p->gapGamma = d.gapGamma;
    p->dynamicAnchorExpansion = d.dynamicAnchorExpansion != 0;
    return p;
}

void pairwiseAlignmentBandingParameters_destruct(PairwiseAlignmentParameters *p) { free(p); }

static int int_member(MiniJson *j, int64_t *out) {
    double v;
    if (minijson_number(j, &v) != 0) return -1;
    *out = (int64_t) v;
    return 0;
}

static int params_member(MiniJson *j, const char *key, void *extra) {
    PairwiseAlignmentParameters *p = extra;
    int b;
    double v;
    if (strcmp(key, "threshold") == 0) return minijson_number(j, &p->threshold);
    if (strcmp(key, "minDiagsBetweenTraceBack") == 0) return int_member(j, &p->minDiagsBetweenTraceBack);
    if (strcmp(key, "traceBackDiagonals") == 0) return int_member(j, &p->traceBackDiagonals);
    if (strcmp(key, "diagonalExpansion") == 0) return int_member(j, &p->diagonalExpansion);
    if (strcmp(key, "constraintDiagonalTrim") == 0) return int_member(j, &p->constraintDiagonalTrim);
    if (strcmp(key, "anchorMatrixBiggerThanThis") == 0) return int_member(j, &p->anchorMatrixBiggerThanThis);
    if (strcmp(key, "repeatMaskMatrixBiggerThanThis") == 0) return int_member(j, &p->repeatMaskMatrixBiggerThanThis);
    if (strcmp(key, "splitMatrixBiggerThanThis") == 0) return int_member(j, &p->splitMatrixBiggerThanThis);
    if (strcmp(key, "alignAmbiguityCharacters") == 0) {
        if (minijson_bool(j, &b) != 0) return -1;
        p->alignAmbiguityCharacters = b != 0;
        return 0;
    }
    if (strcmp(key, "gapGamma") == 0) {
        if (minijson_number(j, &v) != 0) return -1;
        p->gapGamma = (float) v;
        return 0;
    }
    if (strcmp(key, "dynamicAnchorExpansion") == 0) {
        if (minijson_bool(j, &b) != 0) return -1;
        p->dynamicAnchorExpansion = b != 0;
        return 0;
    }
    st_errAbort("ERROR: Unrecognised key in pairwise alignment parameters json: %s\n", key);
    return -1;
}

/* impl/pairwiseAligner.c:1354-1409: defaults for every key that is absent, abort on an unknown key */
PairwiseAlignmentParameters *pairwiseAlignmentParameters_jsonParse(char *buf, size_t r) {
    PairwiseAlignmentParameters *p = pairwiseAlignmentBandingParameters_construct();
    MiniJson j;
    minijson_init(&j, buf, r);
    if (minijson_object(&j, params_member, p) != 0) st_errAbort("ERROR: could not parse pairwise alignment parameters json: %s\n", j.error);
    return p;
}

static void to_engine_params(const PairwiseAlignmentParameters *p, CpbParams *q) {
    memset(q, 0, sizeof(*q));
    q->threshold = p->threshold;
    q->minDiagsBetweenTraceBack = p->minDiagsBetweenTraceBack;
    q->traceBackDiagonals = p->traceBackDiagonals;
    q->diagonalExpansion = p->diagonalExpansion;
    q->constraintDiagonalTrim = p->constraintDiagonalTrim;
    q->anchorMatrixBiggerThanThis = p->anchorMatrixBiggerThanThis;
    q->repeatMaskMatrixBiggerThanThis = p->repeatMaskMatrixBiggerThanThis;
    q->splitMatrixBiggerThanThis = p->splitMatrixBiggerThanThis;
    q->alignAmbiguityCharacters = p->alignAmbiguityCharacters;
    q->gapGamma = p->gapGamma;
    q->dynamicAnchorExpansion = p->dynamicAnchorExpansion;
}

/* --------------------------------------------------------------------------------- device context */

/* The devices this process computes on: one engine context (stream, buffer pools) per GPU, created on first use.  One device by
 * default ($CPECAN_DEVICE or 0); cpecan_setDevices(n) or $CPECAN_DEVICES=n spreads every batch over the first n GPUs.  The library is
 * single threaded towards its callers, as the reference's callers are (SURVEY.md section 8b); inside a call it runs one host thread
 * per device. */
#define CPECAN_MAX_DEVICES 16
static cpb_context *g_ctx[CPECAN_MAX_DEVICES];
static int g_devices[CPECAN_MAX_DEVICES];
static int g_nDevices = 0; /* 0: not chosen yet */
static int64_t g_liveResidentBatches = 0;
static CpecanAnchorProvider g_anchorProvider = NULL;
static void *g_anchorExtra = NULL;

static int any_context(void) {
    for (int i = 0; i < CPECAN_MAX_DEVICES; i++)
        if (g_ctx[i] != NULL) return 1;
    return 0;
}

void cpecan_setDevice(int device) {
    if (any_context() && !(g_nDevices == 1 && g_devices[0] == device)) st_errAbort("cpecan_setDevice: device contexts already exist; call cpecan_shutdown first");
    g_nDevices = 1;
    g_devices[0] = device;
}

void cpecan_setDevices(int n) {
    if (n < 1 || n > CPECAN_MAX_DEVICES) st_errAbort("cpecan_setDevices: %d devices asked for (1 to %d)", n, CPECAN_MAX_DEVICES);
    if (any_context() && g_nDevices != n) st_errAbort("cpecan_setDevices: device contexts already exist; call cpecan_shutdown first");
    g_nDevices = n;
    for (int i = 0; i < n; i++) g_devices[i] = i;
}

void cpecan_setDeviceList(const int *devices, int n) {
    if (n < 1 || n > CPECAN_MAX_DEVICES) st_errAbort("cpecan_setDeviceList: %d devices asked for (1 to %d)", n, CPECAN_MAX_DEVICES);
    if (any_context()) st_errAbort("cpecan_setDeviceList: device contexts already exist; call cpecan_shutdown first");
    g_nDevices = n;
    for (int i = 0; i < n; i++) g_devices[i] = devices[i];
}

int cpecan_getDeviceCount(void) {
    if (g_nDevices == 0) {
        const char *list = getenv("CPECAN_DEVICE_LIST"), *many = getenv("CPECAN_DEVICES"), *one = getenv("CPECAN_DEVICE");
        if (list != NULL && *list != '\0') { /* "0,1,2": explicit ordinals; one may appear twice (two contexts on one GPU, for tests) */
            int devices[CPECAN_MAX_DEVICES], n = 0;
            for (const char *q = list; *q != '\0' && n < CPECAN_MAX_DEVICES;) {
                devices[n++] = atoi(q);
                while (*q != '\0' && *q != ',') q++;
                if (*q == ',') q++;
            }
            cpecan_setDeviceList(devices, n);
        } else if (many != NULL && atoi(many) > 1) {
            cpecan_setDevices(atoi(many));
        } else {
            cpecan_setDevice(one != NULL ? atoi(one) : 0);
        }
    }
    return g_nDevices;
}

void cpecan_shutdown(void) {
    if (g_liveResidentBatches > 0)
        st_errAbort("cpecan_shutdown: %lld resident batches still hold device memory of the contexts; destruct them first", (long long) g_liveResidentBatches);
    for (int i = 0; i < CPECAN_MAX_DEVICES; i++) {
        if (g_ctx[i] != NULL) cpb_context_destroy(g_ctx[i]);
        g_ctx[i] = NULL;
    }
}

void cpecan_setAnchorProvider(CpecanAnchorProvider provider, void *extra) {
    g_anchorProvider = provider;
    g_anchorExtra = extra;
}

/* called from the calling thread only (before the per-device threads start), so creation needs no lock */
static cpb_context *context_of(int slot) {
    cpecan_getDeviceCount();
    if (g_ctx[slot] == NULL) {
        if (cpb_context_create(g_devices[slot], NULL, &g_ctx[slot]) != CPB_OK)
            st_errAbort("cpecan: cannot use CUDA device %d: %s (this library has no CPU implementation of the pair-HMM)", g_devices[slot], cpb_last_error());
    }
    return g_ctx[slot];
}
static cpb_context *context(void) { return context_of(0); }

/* ----------------------------------------------------------------------------- batch marshalling */

typedef struct {
    int64_t n;
    char *seqX, *seqY;
    int64_t *xOff, *yOff, *aOff, *anchors;
    uint8_t *rl, *rr;
} Packed;

static void packed_free(Packed *k) {
    free(k->seqX);
    free(k->seqY);
    free(k->xOff);
    free(k->yOff);
    free(k->aOff);
    free(k->anchors);
    free(k->rl);
    free(k->rr);
}

typedef struct {
    Packed *k;
    const char *const *sX, *const *sY;
    stList *const *anchorPairs;
    int64_t defaultExpansion;
} PackJob;

static void pack_range(int64_t first, int64_t last, void *arg) {
    PackJob *j = arg;
    Packed *k = j->k;
    for (int64_t i = first; i < last; i++) {
        memcpy(k->seqX + k->xOff[i], j->sX[i], (size_t) (k->xOff[i + 1] - k->xOff[i]));
        memcpy(k->seqY + k->yOff[i], j->sY[i], (size_t) (k->yOff[i + 1] - k->yOff[i]));
        const int64_t nA = k->aOff[i + 1] - k->aOff[i];
        for (int64_t a = 0; a < nA; a++) {
            stIntTuple *t = stList_get(j->anchorPairs[i], a);
            int64_t *out = k->anchors + 3 * (k->aOff[i] + a);
            out[0] = stIntTuple_get(t, 0);
            out[1] = stIntTuple_get(t, 1);
            /* anchors are (x, y, expansion); two-element tuples (as the reference's tests build them) use p->diagonalExpansion */
            out[2] = stIntTuple_length(t) > 2 ? stIntTuple_get(t, 2) : j->defaultExpansion;
        }
    }
}

static void pack(Packed *k, int64_t n, const char *const *sX, const char *const *sY, stList *const *anchorPairs, const bool *raggedLeft,
                 const bool *raggedRight, int64_t defaultExpansion) {
    memset(k, 0, sizeof(*k));
    k->n = n;
    k->xOff = cpecan_malloc((size_t) (n + 1) * sizeof(int64_t));
    k->yOff = cpecan_malloc((size_t) (n + 1) * sizeof(int64_t));
    k->aOff = cpecan_malloc((size_t) (n + 1) * sizeof(int64_t));
    k->rl = cpecan_malloc((size_t) n);
    k->rr = cpecan_malloc((size_t) n);
    k->xOff[0] = k->yOff[0] = k->aOff[0] = 0;
    for (int64_t i = 0; i < n; i++) {
        k->xOff[i + 1] = k->xOff[i] + (int64_t) strlen(sX[i]);
        k->yOff[i + 1] = k->yOff[i] + (int64_t) strlen(sY[i]);
        k->aOff[i + 1] = k->aOff[i] + (anchorPairs != NULL && anchorPairs[i] != NULL ? stList_length(anchorPairs[i]) : 0);
        k->rl[i] = raggedLeft != NULL && raggedLeft[i];
        k->rr[i] = raggedRight != NULL && raggedRight[i];
    }
    k->seqX = cpecan_malloc((size_t) k->xOff[n] + 1);
    k->seqY = cpecan_malloc((size_t) k->yOff[n] + 1);
    k->anchors = cpecan_malloc((size_t) (3 * k->aOff[n] + 3) * sizeof(int64_t));
    PackJob job = { k, sX, sY, anchorPairs, defaultExpansion };
    cpecan_parallel_for(n, k->aOff, pack_range, &job);
}

/* runs one engine pass over the packed problems; aborts with the engine's message on failure (the reference has no error codes either) */
/* Page-locked buffers the run fills with the aligned-pair lists while it computes (cpb_batch_set_result_sink): sized by a guess --
 * the reference's threshold keeps about one cell per base -- and simply not used by a run that produces more. */
typedef struct {
    int32_t *tri[3];
    int64_t cap[3];
} Sinks;

static cpb_batch *run(cpb_context *ctx, Packed *k, StateMachine *sM, PairwiseAlignmentParameters *p, int mode, Sinks *sinks) {
    cpb_batch *b = NULL;
    if (cpb_batch_create(ctx, k->n, k->seqX, k->xOff, k->seqY, k->yOff, k->anchors, k->aOff, k->rl, k->rr, &b) != CPB_OK)
        st_errAbort("cpecan: %s", cpb_last_error());
    if (sinks != NULL) {
        const int nLists = mode == CPB_MODE_ALIGNED_PAIRS ? 1 : (mode == CPB_MODE_ALIGNED_PAIRS_INDELS ? 3 : 0);
        for (int l = 0; l < nLists; l++) {
            sinks->cap[l] = 2 * (k->xOff[k->n] < k->yOff[k->n] ? k->xOff[k->n] : k->yOff[k->n]) + 4096;
            sinks->tri[l] = cpb_pinned_alloc(ctx, (size_t) sinks->cap[l] * 3 * sizeof(int32_t));
            if (sinks->tri[l] != NULL) cpb_batch_set_result_sink(b, l, sinks->tri[l], sinks->cap[l]);
        }
    }
    CpbParams q;
    to_engine_params(p, &q);
    const int rc = cpb_batch_run(b, cpecan_model_of(sM), &q, mode);
    if (rc == CPB_ERR_BAND) st_errAbort("%s: %s", PAIRWISE_ALIGNMENT_EXCEPTION_ID, cpb_last_error());
    if (rc != CPB_OK) st_errAbort("cpecan: %s", cpb_last_error());
    return b;
}

/* list `which` of the last run as n stLists of (pInt, x, y) tuples */
typedef struct {
    stList **lists;
    const int64_t *off;
    const int32_t *tri;
} ListJob;

static void lists_range(int64_t first, int64_t last, void *arg) {
    ListJob *j = arg;
    for (int64_t i = first; i < last; i++) j->lists[i] = cpecan_tripleList_construct(j->tri + 3 * j->off[i], j->off[i + 1] - j->off[i]);
}

static stList **fetch_lists(cpb_context *ctx, cpb_batch *b, int64_t n, int which, Sinks *sinks) {
    const int64_t total = cpb_batch_result_count(b, which);
    int64_t *off = cpecan_malloc((size_t) (n + 1) * sizeof(int64_t));
    const size_t triBytes = (size_t) (3 * total + 3) * sizeof(int32_t);
    /* the sink the run filled, if the list fitted; else page-locked staging from the context's pool; pageable memory if there is none */
    int32_t *tri = sinks != NULL && sinks->tri[which] != NULL && total <= sinks->cap[which] ? sinks->tri[which] : NULL;
    const int fromSink = tri != NULL;
    if (!fromSink) tri = cpb_pinned_alloc(ctx, triBytes);
    const int pinned = tri != NULL;
    if (!pinned) tri = cpecan_malloc(triBytes);
    /* same list order as the reference's own lists (its callers may depend on it, e.g. the MEA walk-back) */
    const int timing = getenv("CPECAN_HOST_TIMING") != NULL;
    double t0 = timing ? wall_seconds() : 0.0;
    if (cpb_batch_fetch_pairs_reference_order(b, which, off, tri) != CPB_OK) st_errAbort("cpecan: %s", cpb_last_error());
    if (timing) fprintf(stderr, "    copy + reference order of %lld triples %8.1f ms\n", (long long) total, 1e3 * (wall_seconds() - t0));
    stList **lists = cpecan_malloc((size_t) (n > 0 ? n : 1) * sizeof(stList *));
    ListJob job = { lists, off, tri };
    t0 = timing ? wall_seconds() : 0.0;
    cpecan_parallel_for(n, off, lists_range, &job);
    if (timing) fprintf(stderr, "    lists of slab tuples               %8.1f ms\n", 1e3 * (wall_seconds() - t0));
    free(off);
    if (fromSink) { /* released with the other sinks */
    } else if (pinned) {
        cpb_pinned_free(ctx, tri);
    } else {
        free(tri);
    }
    return lists;
}

/* ------------------------------------------------------------------------------- batched entries */

/*
 * One batch over the device set.  Problems are independent, so they are dealt to the devices by longest-processing-time-first on an
 * estimate of their band cells (diagonals x (mean anchor gap + expansion)): the most expensive problem goes to the least loaded
 * device, and so on down the list.  Every device then gets one host thread that marshals its share, runs the engine pass on its own
 * context and stream, and writes its results into the caller's arrays at the problems' own indices -- no data-path traffic between
 * GPUs.  The only exchange is the EM reduction of the expectation totals (cpb_expectations_allreduce, NCCL).
 */
typedef struct {
    int slot;
    cpb_context *ctx;
    int64_t n;          /* problems of this device */
    const int64_t *idx; /* their indices in the caller's arrays, ascending */
    /* the call */
    StateMachine *sM;
    PairwiseAlignmentParameters *p;
    int mode, reweight, keepBatch;
    double gapGamma;
    const char *const *sX, *const *sY;
    stList *const *anchorPairs;
    const bool *raggedLeft, *raggedRight;
    /* results, in the caller's indexing */
    stList **lists[3];
    double *logProbs;
    cpb_batch *batch; /* expectation mode / keepBatch: left alive for the reduction */
} DeviceJob;

static void *device_job(void *v) {
    DeviceJob *j = v;
    const int64_t n = j->n;
    const int timing = getenv("CPECAN_HOST_TIMING") != NULL; /* stage times of the marshalling on stderr */
    double t0 = wall_seconds(), t1;
#define STAGE(what)                                                                                          \
    if (timing) {                                                                                            \
        t1 = wall_seconds();                                                                                 \
        fprintf(stderr, "  [cpecan device %d] %-28s %8.1f ms\n", g_devices[j->slot], what, 1e3 * (t1 - t0)); \
        t0 = t1;                                                                                             \
    }
    const char **sX = cpecan_malloc((size_t) (n + 1) * sizeof(char *)), **sY = cpecan_malloc((size_t) (n + 1) * sizeof(char *));
    stList **an = cpecan_malloc((size_t) (n + 1) * sizeof(stList *));
    bool *rl = cpecan_malloc((size_t) n + 1), *rr = cpecan_malloc((size_t) n + 1);
    for (int64_t i = 0; i < n; i++) {
        const int64_t g = j->idx != NULL ? j->idx[i] : i;
        sX[i] = j->sX[g];
        sY[i] = j->sY[g];
        an[i] = j->anchorPairs != NULL ? j->anchorPairs[g] : NULL;
        rl[i] = j->raggedLeft != NULL && j->raggedLeft[g];
        rr[i] = j->raggedRight != NULL && j->raggedRight[g];
    }
    Packed k;
    Sinks sinks;
    memset(&sinks, 0, sizeof(sinks));
    pack(&k, n, sX, sY, an, rl, rr, j->p->diagonalExpansion);
    STAGE("pack (tuples -> flat arrays)");
    cpb_batch *b = NULL;
    if (j->mode < 0) { /* resident batch: inputs to the device, no run yet */
        if (cpb_batch_create(j->ctx, k.n, k.seqX, k.xOff, k.seqY, k.yOff, k.anchors, k.aOff, k.rl, k.rr, &b) != CPB_OK) st_errAbort("cpecan: %s", cpb_last_error());
    } else {
        b = run(j->ctx, &k, j->sM, j->p, j->mode, j->reweight ? NULL : &sinks); /* (reweighting rewrites the list on the device after the run) */
    }
    STAGE("device pass (create + run)");
    if (j->mode == CPB_MODE_ALIGNED_PAIRS || j->mode == CPB_MODE_ALIGNED_PAIRS_INDELS) {
        if (j->reweight && cpb_batch_reweight_pairs(b, j->gapGamma) != CPB_OK) st_errAbort("cpecan: %s", cpb_last_error());
        const int nLists = j->mode == CPB_MODE_ALIGNED_PAIRS ? 1 : 3;
        for (int l = 0; l < nLists; l++) {
            stList **mine = fetch_lists(j->ctx, b, n, l, &sinks);
            for (int64_t i = 0; i < n; i++) j->lists[l][j->idx != NULL ? j->idx[i] : i] = mine[i];
            free(mine);
        }
    } else if (j->mode == CPB_MODE_FORWARD) {
        double *lp = cpecan_malloc((size_t) (n + 1) * sizeof(double));
        if (cpb_batch_fetch_forward(b, lp) != CPB_OK) st_errAbort("cpecan: %s", cpb_last_error());
        for (int64_t i = 0; i < n; i++) j->logProbs[j->idx != NULL ? j->idx[i] : i] = lp[i];
        free(lp);
    }
    for (int l = 0; l < 3; l++)
        if (sinks.tri[l] != NULL) cpb_pinned_free(j->ctx, sinks.tri[l]);
    STAGE("fetch (copy, order, lists)");
    if (j->mode == CPB_MODE_EXPECTATIONS || j->keepBatch) j->batch = b;
    else cpb_batch_destroy(b);
    packed_free(&k);
    free(sX);
    free(sY);
    free(an);
    free(rl);
    free(rr);
    STAGE("release");
#undef STAGE
    return NULL;
}

/* longest-processing-time-first: idx[d] / count[d] = the problems of device d, ascending */
typedef struct {
    int64_t cost, index;
} CostItem;
static int cost_descending(const void *a, const void *b) {
    const CostItem *x = a, *y = b;
    if (x->cost != y->cost) return x->cost > y->cost ? -1 : 1;
    return x->index < y->index ? -1 : (x->index > y->index ? 1 : 0);
}
static int index_ascending(const void *a, const void *b) {
    const int64_t x = *(const int64_t *) a, y = *(const int64_t *) b;
    return x < y ? -1 : (x > y ? 1 : 0);
}
static void deal_problems(int64_t n, const char *const *sX, const char *const *sY, stList *const *anchorPairs, int64_t expansion, int nDev, int64_t **idx,
                          int64_t *count) {
    CostItem *items = cpecan_malloc((size_t) (n + 1) * sizeof(CostItem));
    for (int64_t i = 0; i < n; i++) {
        const int64_t lX = (int64_t) strlen(sX[i]), lY = (int64_t) strlen(sY[i]);
        const int64_t nA = anchorPairs != NULL && anchorPairs[i] != NULL ? stList_length(anchorPairs[i]) : 0;
        int64_t gap = (lX + lY) / (2 * (nA + 1)), cap = (lX < lY ? lX : lY) + 1;
        if (gap > cap) gap = cap;
        items[i].cost = (lX + lY + 1) * (gap + expansion + 1);
        items[i].index = i;
    }
    qsort(items, (size_t) n, sizeof(CostItem), cost_descending);
    int64_t load[CPECAN_MAX_DEVICES];
    for (int d = 0; d < nDev; d++) {
        idx[d] = cpecan_malloc((size_t) (n + 1) * sizeof(int64_t));
        count[d] = 0;
        load[d] = 0;
    }
    for (int64_t i = 0; i < n; i++) {
        int best = 0;
        for (int d = 1; d < nDev; d++)
            if (load[d] < load[best]) best = d;
        idx[best][count[best]++] = items[i].index;
        load[best] += items[i].cost;
    }
    for (int d = 0; d < nDev; d++) qsort(idx[d], (size_t) count[d], sizeof(int64_t), index_ascending);
    free(items);
}

/* runs `proto` (the call's arguments) over the device set; jobs[] keeps the per-device state for the caller (batches of expectation runs) */
static int run_on_devices(DeviceJob *proto, int64_t n, DeviceJob *jobs, int64_t **idxOut) {
    const int nDev = (int) (cpecan_getDeviceCount() < n ? cpecan_getDeviceCount() : (n > 0 ? n : 1));
    int64_t *idx[CPECAN_MAX_DEVICES], count[CPECAN_MAX_DEVICES];
    if (nDev <= 1) {
        jobs[0] = *proto;
        jobs[0].slot = 0;
        jobs[0].ctx = context_of(0);
        jobs[0].n = n;
        jobs[0].idx = NULL;
        device_job(&jobs[0]);
        if (idxOut != NULL) idxOut[0] = NULL;
        return 1;
    }
    deal_problems(n, proto->sX, proto->sY, proto->anchorPairs, proto->p->diagonalExpansion, nDev, idx, count);
    pthread_t ids[CPECAN_MAX_DEVICES];
    for (int d = 0; d < nDev; d++) {
        jobs[d] = *proto;
        jobs[d].slot = d;
        jobs[d].ctx = context_of(d); /* created here, in the calling thread */
        jobs[d].n = count[d];
        jobs[d].idx = idx[d];
    }
    for (int d = 0; d < nDev; d++)
        if (pthread_create(&ids[d], NULL, device_job, &jobs[d]) != 0) st_errAbort("cpecan: cannot start the host thread of device %d", g_devices[d]);
    for (int d = 0; d < nDev; d++) pthread_join(ids[d], NULL);
    for (int d = 0; d < nDev; d++) {
        if (idxOut != NULL) idxOut[d] = idx[d];
        else free(idx[d]);
    }
    return nDev;
}

static DeviceJob job_of(StateMachine *sM, const char *const *sX, const char *const *sY, stList *const *anchorPairs, PairwiseAlignmentParameters *p,
                        const bool *raggedLeft, const bool *raggedRight, int mode) {
    DeviceJob j;
    memset(&j, 0, sizeof(j));
    j.sM = sM;
    j.p = p;
    j.mode = mode;
    j.sX = sX;
    j.sY = sY;
    j.anchorPairs = anchorPairs;
    j.raggedLeft = raggedLeft;
    j.raggedRight = raggedRight;
    return j;
}

static stList **new_list_array(int64_t n) {
    stList **l = cpecan_malloc((size_t) (n > 0 ? n : 1) * sizeof(stList *));
    memset(l, 0, (size_t) (n > 0 ? n : 1) * sizeof(stList *));
    return l;
}

stList **getAlignedPairsUsingAnchorsBatch(StateMachine *sM, int64_t n, const char *const *sX, const char *const *sY,
                                          stList *const *anchorPairs, PairwiseAlignmentParameters *p, const bool *raggedLeft,
                                          const bool *raggedRight) {
    DeviceJob proto = job_of(sM, sX, sY, anchorPairs, p, raggedLeft, raggedRight, CPB_MODE_ALIGNED_PAIRS), jobs[CPECAN_MAX_DEVICES];
    proto.lists[0] = new_list_array(n);
    run_on_devices(&proto, n, jobs, NULL);
    return proto.lists[0];
}

stList **getReweightedAlignedPairsUsingAnchorsBatch(StateMachine *sM, int64_t n, const char *const *sX, const char *const *sY,
                                                    stList *const *anchorPairs, PairwiseAlignmentParameters *p, const bool *raggedLeft,
                                                    const bool *raggedRight, double gapGamma) {
    DeviceJob proto = job_of(sM, sX, sY, anchorPairs, p, raggedLeft, raggedRight, CPB_MODE_ALIGNED_PAIRS), jobs[CPECAN_MAX_DEVICES];
    proto.lists[0] = new_list_array(n);
    proto.reweight = 1;
    proto.gapGamma = gapGamma;
    run_on_devices(&proto, n, jobs, NULL);
    return proto.lists[0];
}

void getAlignedPairsWithIndelsUsingAnchorsBatch(StateMachine *sM, int64_t n, const char *const *sX, const char *const *sY,
                                                stList *const *anchorPairs, PairwiseAlignmentParameters *p, stList ***alignedPairs,
                                                stList ***gapXPairs, stList ***gapYPairs, const bool *raggedLeft, const bool *raggedRight) {
    DeviceJob proto = job_of(sM, sX, sY, anchorPairs, p, raggedLeft, raggedRight, CPB_MODE_ALIGNED_PAIRS_INDELS), jobs[CPECAN_MAX_DEVICES];
    for (int l = 0; l < 3; l++) proto.lists[l] = new_list_array(n);
    run_on_devices(&proto, n, jobs, NULL);
    *alignedPairs = proto.lists[0];
    *gapXPairs = proto.lists[1];
    *gapYPairs = proto.lists[2];
}

/* the expectation totals of nDev finished expectation runs, summed: NCCL all-reduce across the devices when there are several (every
 * device then holds the sum; device 0's copy is read), else the one total as it is */
static void add_expectations(Hmm *hmmExpectations, int64_t S, cpb_batch **batches, int nDev) {
    double total[CPB_HMM_LEN(5)];
    if (nDev > 1 && cpb_expectations_allreduce(batches, nDev) != CPB_OK) {
        /* no NCCL in this process: the 58 / 106 doubles per device are added up here instead (in device order) */
        static int told = 0;
        if (!told) fprintf(stderr, "cpecan: %s; summing the expectation totals of the %d devices on the host\n", cpb_last_error(), nDev);
        told = 1;
        double part[CPB_HMM_LEN(5)];
        memset(total, 0, sizeof(total));
        for (int d = 0; d < nDev; d++) {
            if (cpb_batch_fetch_expectations(batches[d], NULL, part) != CPB_OK) st_errAbort("cpecan: %s", cpb_last_error());
            for (int64_t i = 0; i < CPB_HMM_LEN(S); i++) total[i] += part[i];
        }
    } else if (cpb_batch_fetch_expectations(batches[0], NULL, total) != CPB_OK) {
        st_errAbort("cpecan: %s", cpb_last_error());
    }
    for (int64_t i = 0; i < S * S; i++) hmmExpectations->transitions[i] += total[i];
    for (int64_t i = 0; i < S * 16; i++) hmmExpectations->emissions[i] += total[S * S + i];
    hmmExpectations->likelihood += total[S * S + S * 16];
}

void getExpectationsUsingAnchorsBatch(StateMachine *sM, Hmm *hmmExpectations, int64_t n, const char *const *sX, const char *const *sY,
                                      stList *const *anchorPairs, PairwiseAlignmentParameters *p, const bool *raggedLeft,
                                      const bool *raggedRight) {
    if (hmmExpectations->stateNumber != sM->stateNumber)
        st_errAbort("getExpectations: the Hmm has %lld states, the state machine %lld", (long long) hmmExpectations->stateNumber,
                    (long long) sM->stateNumber);
    DeviceJob proto = job_of(sM, sX, sY, anchorPairs, p, raggedLeft, raggedRight, CPB_MODE_EXPECTATIONS), jobs[CPECAN_MAX_DEVICES];
    const int nDev = run_on_devices(&proto, n, jobs, NULL);
    cpb_batch *batches[CPECAN_MAX_DEVICES];
    for (int d = 0; d < nDev; d++) batches[d] = jobs[d].batch;
    add_expectations(hmmExpectations, sM->stateNumber, batches, nDev);
    for (int d = 0; d < nDev; d++) cpb_batch_destroy(batches[d]);
}

/* ---- resident batches: the inputs go to the devices once, every EM iteration is one more pass with a new model ---- */

struct _cpecanResidentBatch {
    cpb_batch *b[CPECAN_MAX_DEVICES];
    int nDev;
    int64_t n;
};

CpecanResidentBatch *cpecanResidentBatch_construct(int64_t n, const char *const *sX, const char *const *sY, stList *const *anchorPairs,
                                                   PairwiseAlignmentParameters *p, const bool *raggedLeft, const bool *raggedRight) {
    DeviceJob proto = job_of(NULL, sX, sY, anchorPairs, p, raggedLeft, raggedRight, -1), jobs[CPECAN_MAX_DEVICES];
    proto.keepBatch = 1;
    CpecanResidentBatch *r = cpecan_malloc(sizeof(*r));
    memset(r, 0, sizeof(*r));
    r->n = n;
    r->nDev = run_on_devices(&proto, n, jobs, NULL);
    for (int d = 0; d < r->nDev; d++) r->b[d] = jobs[d].batch;
    g_liveResidentBatches++;
    return r;
}

void cpecanResidentBatch_destruct(CpecanResidentBatch *r) {
    if (r == NULL) return;
    for (int d = 0; d < r->nDev; d++) cpb_batch_destroy(r->b[d]);
    g_liveResidentBatches--;
    free(r);
}

typedef struct {
    cpb_batch *b;
    const CpbModel *model;
    const CpbParams *q;
    int updateAnchors; /* 0: an expectation run; 1: realign and re-anchor (cpecanResidentBatch_updateAnchors) */
    float matchGamma;
} ResidentRun;
static void resident_check(int rc) {
    if (rc == CPB_ERR_BAND) st_errAbort("%s: %s", PAIRWISE_ALIGNMENT_EXCEPTION_ID, cpb_last_error());
    if (rc != CPB_OK) st_errAbort("cpecan: %s", cpb_last_error());
}
static void *resident_run(void *v) {
    ResidentRun *r = v;
    if (!r->updateAnchors) {
        resident_check(cpb_batch_run(r->b, r->model, r->q, CPB_MODE_EXPECTATIONS));
        return NULL;
    }
    /* cPecanRealign's default steps for every alignment (job_finish: reweight, ordered chain), then the anchors job_prepare makes from the
     * cigar it would write; no list leaves the device */
    resident_check(cpb_batch_run(r->b, r->model, r->q, CPB_MODE_ALIGNED_PAIRS));
    resident_check(cpb_batch_reweight_pairs(r->b, r->q->gapGamma));
    resident_check(cpb_batch_ordered_chain(r->b, r->matchGamma));
    resident_check(cpb_batch_anchors_from_alignments(r->b, r->q));
    return NULL;
}

/* one host thread per device */
static void resident_each(CpecanResidentBatch *r, StateMachine *sM, const CpbParams *q, int updateAnchors, float matchGamma) {
    ResidentRun runs[CPECAN_MAX_DEVICES];
    pthread_t ids[CPECAN_MAX_DEVICES];
    for (int d = 0; d < r->nDev; d++) {
        runs[d].b = r->b[d];
        runs[d].model = cpecan_model_of(sM);
        runs[d].q = q;
        runs[d].updateAnchors = updateAnchors;
        runs[d].matchGamma = matchGamma;
    }
    if (r->nDev == 1) {
        resident_run(&runs[0]);
    } else {
        for (int d = 0; d < r->nDev; d++)
            if (pthread_create(&ids[d], NULL, resident_run, &runs[d]) != 0) st_errAbort("cpecan: cannot start a host thread");
        for (int d = 0; d < r->nDev; d++) pthread_join(ids[d], NULL);
    }
}

void cpecanResidentBatch_getExpectations(CpecanResidentBatch *r, StateMachine *sM, Hmm *hmmExpectations, PairwiseAlignmentParameters *p) {
    if (hmmExpectations->stateNumber != sM->stateNumber)
        st_errAbort("getExpectations: the Hmm has %lld states, the state machine %lld", (long long) hmmExpectations->stateNumber,
                    (long long) sM->stateNumber);
    CpbParams q;
    to_engine_params(p, &q);
    resident_each(r, sM, &q, 0, 0.0f);
    add_expectations(hmmExpectations, sM->stateNumber, r->b, r->nDev);
}

void cpecanResidentBatch_updateAnchors(CpecanResidentBatch *r, StateMachine *sM, PairwiseAlignmentParameters *p, float matchGamma) {
    if (!(matchGamma >= 0.0f && matchGamma <= 1.0f)) st_errAbort("cpecanResidentBatch_updateAnchors: matchGamma must be in [0, 1], not %g", (double) matchGamma);
    CpbParams q;
    to_engine_params(p, &q);
    resident_each(r, sM, &q, 1, matchGamma);
}

void computeForwardProbabilityBatch(StateMachine *sM, int64_t n, const char *const *sX, const char *const *sY, stList *const *anchorPairs,
                                    PairwiseAlignmentParameters *p, const bool *raggedLeft, const bool *raggedRight, double *logProbs) {
    DeviceJob proto = job_of(sM, sX, sY, anchorPairs, p, raggedLeft, raggedRight, CPB_MODE_FORWARD), jobs[CPECAN_MAX_DEVICES];
    proto.logProbs = logProbs;
    run_on_devices(&proto, n, jobs, NULL);
}

/* ---------------------------------------------------------------- the reference's one-pair forms */

stList *getAlignedPairsUsingAnchors(StateMachine *sM, const char *sX, const char *sY, stList *anchorPairs, PairwiseAlignmentParameters *p,
                                    bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd) {
    stList **lists = getAlignedPairsUsingAnchorsBatch(sM, 1, &sX, &sY, &anchorPairs, p, &alignmentHasRaggedLeftEnd, &alignmentHasRaggedRightEnd);
    stList *out = lists[0];
    free(lists);
    return out;
}

void getAlignedPairsWithIndelsUsingAnchors(StateMachine *sM, const char *sX, const char *sY, stList *anchorPairs,
                                           PairwiseAlignmentParameters *p, stList **alignedPairs, stList **gapXPairs, stList **gapYPairs,
                                           bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd) {
    stList **m, **gx, **gy;
    getAlignedPairsWithIndelsUsingAnchorsBatch(sM, 1, &sX, &sY, &anchorPairs, p, &m, &gx, &gy, &alignmentHasRaggedLeftEnd,
                                               &alignmentHasRaggedRightEnd);
    *alignedPairs = m[0];
    *gapXPairs = gx[0];
    *gapYPairs = gy[0];
    free(m);
    free(gx);
    free(gy);
}

void getExpectationsUsingAnchors(StateMachine *sM, Hmm *hmmExpectations, const char *sX, const char *sY, stList *anchorPairs,
                                 PairwiseAlignmentParameters *p, bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd) {
    getExpectationsUsingAnchorsBatch(sM, hmmExpectations, 1, &sX, &sY, &anchorPairs, p, &alignmentHasRaggedLeftEnd, &alignmentHasRaggedRightEnd);
}

double computeForwardProbability(char *seqX, char *seqY, stList *anchorPairs, PairwiseAlignmentParameters *p, StateMachine *sM,
                                 bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd) {
    const char *sX = seqX, *sY = seqY;
    double v = 0.0;
    computeForwardProbabilityBatch(sM, 1, &sX, &sY, &anchorPairs, p, &alignmentHasRaggedLeftEnd, &alignmentHasRaggedRightEnd, &v);
    return v;
}

/* anchors for the forms that take none (getBlastPairsForPairwiseAlignmentParameters, impl/pairwiseAligner.c:1162-1196) */
static stList *anchors_for(const char *sX, const char *sY, PairwiseAlignmentParameters *p) {
    const int64_t lX = (int64_t) strlen(sX), lY = (int64_t) strlen(sY);
    if (g_anchorProvider != NULL && lX * lY > p->anchorMatrixBiggerThanThis) return g_anchorProvider(sX, sY, lX, lY, p, g_anchorExtra);
    return getBlastPairsForPairwiseAlignmentParameters(sX, sY, lX, lY, p);
}

/* anchors of many problems on the host threads, then ONE device pass: what makeAllPairwiseAlignments' loop (impl/multipleAligner.c:
 * 653-681: getAlignedPairs per pair of sequences) becomes */
typedef struct {
    const char *const *sX, *const *sY;
    PairwiseAlignmentParameters *p;
    stList **anchors;
} AnchorJob;
static void anchors_range(int64_t first, int64_t last, void *arg) {
    AnchorJob *j = arg;
    for (int64_t i = first; i < last; i++) j->anchors[i] = anchors_for(j->sX[i], j->sY[i], j->p);
}
stList **getAlignedPairsBatch(StateMachine *sM, int64_t n, const char *const *sX, const char *const *sY, PairwiseAlignmentParameters *p,
                              const bool *raggedLeft, const bool *raggedRight) {
    stList **anchors = new_list_array(n);
    int64_t *weight = cpecan_malloc((size_t) (n + 1) * sizeof(int64_t)); /* anchoring costs about the sequence length */
    weight[0] = 0;
    for (int64_t i = 0; i < n; i++) weight[i + 1] = weight[i] + (int64_t) strlen(sX[i]) + (int64_t) strlen(sY[i]) + 1;
    AnchorJob job = { sX, sY, p, anchors };
    cpecan_parallel_for(n, weight, anchors_range, &job);
    free(weight);
    stList **out = getAlignedPairsUsingAnchorsBatch(sM, n, sX, sY, anchors, p, raggedLeft, raggedRight);
    for (int64_t i = 0; i < n; i++) stList_destruct(anchors[i]);
    free(anchors);
    return out;
}

stList *getAlignedPairs(StateMachine *sM, const char *string1, const char *string2, PairwiseAlignmentParameters *p,
                        bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd) {
    stList *anchorPairs = anchors_for(string1, string2, p);
    stList *out = getAlignedPairsUsingAnchors(sM, string1, string2, anchorPairs, p, alignmentHasRaggedLeftEnd, alignmentHasRaggedRightEnd);
    stList_destruct(anchorPairs);
    return out;
}

void getAlignedPairsWithIndels(StateMachine *sM, const char *string1, const char *string2, PairwiseAlignmentParameters *p,
                               stList **alignedPairs, stList **gapXPairs, stList **gapYPairs, bool alignmentHasRaggedLeftEnd,
                               bool alignmentHasRaggedRightEnd) {
    stList *anchorPairs = anchors_for(string1, string2, p);
    getAlignedPairsWithIndelsUsingAnchors(sM, string1, string2, anchorPairs, p, alignedPairs, gapXPairs, gapYPairs, alignmentHasRaggedLeftEnd,
                                          alignmentHasRaggedRightEnd);
    stList_destruct(anchorPairs);
}

void getExpectations(StateMachine *sM, Hmm *hmmExpectations, const char *sX, const char *sY, PairwiseAlignmentParameters *p,
                     bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd) {
    stList *anchorPairs = anchors_for(sX, sY, p);
    getExpectationsUsingAnchors(sM, hmmExpectations, sX, sY, anchorPairs, p, alignmentHasRaggedLeftEnd, alignmentHasRaggedRightEnd);
    stList_destruct(anchorPairs);
}

/* ------------------------------------------------------------------------ test-visible helpers */

Diagonal diagonal_construct(int64_t xay, int64_t xmyL, int64_t xmyR) {
    /* impl/pairwiseAligner.c:30-43: both ends share the parity of xay and xmyL <= xmyR */
    if ((xay + xmyL) % 2 != 0 || (xay + xmyR) % 2 != 0 || xmyL > xmyR)
        st_errAbort("%s: Attempt to create diagonal with invalid coordinates: xay %lld xmyL %lld xmyR %lld", PAIRWISE_ALIGNMENT_EXCEPTION_ID,
                    (long long) xay, (long long) xmyL, (long long) xmyR);
    Diagonal d = { xay, xmyL, xmyR };
    return d;
}
int64_t diagonal_getXay(Diagonal d) { return d.xay; }
int64_t diagonal_getMinXmy(Diagonal d) { return d.xmyL; }
int64_t diagonal_getMaxXmy(Diagonal d) { return d.xmyR; }
int64_t diagonal_getWidth(Diagonal d) { return (d.xmyR - d.xmyL) / 2 + 1; }
int64_t diagonal_getXCoordinate(int64_t xay, int64_t xmy) { return (xay + xmy) / 2; }
int64_t diagonal_getYCoordinate(int64_t xay, int64_t xmy) { return (xay - xmy) / 2; }
int64_t diagonal_equals(Diagonal d1, Diagonal d2) { return d1.xay == d2.xay && d1.xmyL == d2.xmyL && d1.xmyR == d2.xmyR; }

struct _band {
    Diagonal *diagonals;
    int64_t lXalY; /* lX + lY: diagonals 0 .. lXalY */
};
struct _bandIterator {
    Band *band;
    int64_t index;
};

static Band *band_from_device(stList *anchorPairs, int64_t lX, int64_t lY, int64_t expansion, int dynamic) {
    const int64_t nA = anchorPairs != NULL ? stList_length(anchorPairs) : 0;
    int64_t *an = cpecan_malloc((size_t) (3 * nA + 3) * sizeof(int64_t));
    for (int64_t i = 0; i < nA; i++) {
        stIntTuple *t = stList_get(anchorPairs, i);
        an[3 * i] = stIntTuple_get(t, 0);
        an[3 * i + 1] = stIntTuple_get(t, 1);
        an[3 * i + 2] = stIntTuple_length(t) > 2 ? stIntTuple_get(t, 2) : expansion;
    }
    int64_t *out3 = cpecan_malloc((size_t) (3 * (lX + lY + 1)) * sizeof(int64_t));
    const int rc = cpb_band(context(), an, nA, lX, lY, expansion, dynamic, out3);
    if (rc == CPB_ERR_BAND) st_errAbort("%s: %s", PAIRWISE_ALIGNMENT_EXCEPTION_ID, cpb_last_error());
    if (rc != CPB_OK) st_errAbort("cpecan: %s", cpb_last_error());
    Band *band = cpecan_malloc(sizeof(*band));
    band->lXalY = lX + lY;
    band->diagonals = cpecan_malloc((size_t) (lX + lY + 1) * sizeof(Diagonal));
    for (int64_t d = 0; d <= lX + lY; d++) {
        band->diagonals[d].xay = out3[3 * d];
        band->diagonals[d].xmyL = out3[3 * d + 1];
        band->diagonals[d].xmyR = out3[3 * d + 2];
    }
    free(an);
    free(out3);
    return band;
}

Band *band_construct(stList *anchorPairs, int64_t lX, int64_t lY, int64_t expansion) { return band_from_device(anchorPairs, lX, lY, expansion, 0); }
Band *band_constructDynamic(stList *anchorPairs, int64_t lX, int64_t lY) { return band_from_device(anchorPairs, lX, lY, 0, 1); }

void band_destruct(Band *band) {
    if (band == NULL) return;
    free(band->diagonals);
    free(band);
}

BandIterator *bandIterator_construct(Band *band) {
    BandIterator *it = cpecan_malloc(sizeof(*it));
    it->band = band;
    it->index = 0;
    return it;
}
BandIterator *bandIterator_clone(BandIterator *bandIterator) {
    BandIterator *it = cpecan_malloc(sizeof(*it));
    *it = *bandIterator;
    return it;
}
void bandIterator_destruct(BandIterator *bandIterator) { free(bandIterator); }

/* impl/pairwiseAligner.c:263-277: the index runs over [0, lX+lY+1]; reads clamp to the first / last diagonal */
Diagonal bandIterator_getNext(BandIterator *it) {
    const int64_t last = it->band->lXalY;
    Diagonal d = it->band->diagonals[it->index > last ? last : it->index];
    if (it->index <= last) it->index++;
    return d;
}
Diagonal bandIterator_getPrevious(BandIterator *it) {
    if (it->index > 0) it->index--;
    return it->band->diagonals[it->index];
}

Symbol symbol_convertCharToSymbol(char i) {
    switch (i) {
    case 'A':
    case 'a':
        return a;
    case 'C':
    case 'c':
        return c;
    case 'G':
    case 'g':
        return g;
    case 'T':
    case 't':
        return t;
    default:
        return n;
    }
}

char symbol_convertSymbolToChar(Symbol i) {
    static const char letters[] = "ACGTN";
    return letters[(int) i >= 0 && (int) i < 4 ? (int) i : 4];
}

Symbol *symbol_convertStringToSymbols(const char *s, int64_t sL) {
    Symbol *out = cpecan_malloc((size_t) (sL > 0 ? sL : 1) * sizeof(Symbol));
    for (int64_t i = 0; i < sL; i++) out[i] = symbol_convertCharToSymbol(s[i]);
    return out;
}

stList *getSplitPoints(stList *anchorPairs, int64_t lX, int64_t lY, int64_t maxMatrixSize, bool alignmentHasRaggedLeftEnd,
                       bool alignmentHasRaggedRightEnd) {
    const int64_t nA = anchorPairs != NULL ? stList_length(anchorPairs) : 0;
    int64_t *an = cpecan_malloc((size_t) (3 * nA + 3) * sizeof(int64_t));
    for (int64_t i = 0; i < nA; i++) {
        stIntTuple *t = stList_get(anchorPairs, i);
        an[3 * i] = stIntTuple_get(t, 0);
        an[3 * i + 1] = stIntTuple_get(t, 1);
        an[3 * i + 2] = 0;
    }
    int64_t cap = nA + 2;
    int64_t *out4 = cpecan_malloc((size_t) (4 * cap) * sizeof(int64_t));
    const int64_t nReg = cpb_split_points(an, nA, lX, lY, maxMatrixSize, alignmentHasRaggedLeftEnd, alignmentHasRaggedRightEnd, out4, cap);
    if (nReg < 0 || nReg > cap) st_errAbort("cpecan: getSplitPoints failed: %s", cpb_last_error());
    stList *out = stList_construct3(0, (void (*)(void *)) stIntTuple_destruct);
    for (int64_t r = 0; r < nReg; r++) stList_append(out, stIntTuple_construct4(out4[4 * r], out4[4 * r + 1], out4[4 * r + 2], out4[4 * r + 3]));
    free(an);
    free(out4);
    return out;
}
