/*
 * cpecan_b200.h -- flat C-ABI of the B200-native pair-HMM engine (libcpecan_b200.so).
 *
 * This is the batched boundary below cPecan's one-pair-per-call C API.  Every entry point takes plain
 * pointers and sizes (no sonLib, no torch types); the reference-compatible wrappers declared in
 * include/cpecan/pairwiseAligner.h (getAlignedPairsUsingAnchors, getExpectationsUsingAnchors, ...)
 * are thin adaptors over these, and INTEGRATION.md shows the binding a cPecan maintainer would add.
 *
 * Reference interfaces replaced (all paths relative to the cPecan tree):
 *   cpb_batch_run(CPB_MODE_ALIGNED_PAIRS)        getAlignedPairsUsingAnchors            impl/pairwiseAligner.c:1431
 *   cpb_batch_run(CPB_MODE_ALIGNED_PAIRS_INDELS) getAlignedPairsWithIndelsUsingAnchors  impl/pairwiseAligner.c:1451
 *   cpb_batch_run(CPB_MODE_EXPECTATIONS)         getExpectationsUsingAnchors            impl/pairwiseAligner.c:1500
 *   cpb_batch_run(CPB_MODE_FORWARD)              computeForwardProbability              impl/pairwiseAligner.c:936
 *   cpb_params_default                           pairwiseAlignmentBandingParameters_construct  :1334
 *   cpb_model_default / cpb_model_from_hmm       stateMachine5_construct / stateMachine3_construct /
 *                                                hmm_getStateMachine                    impl/stateMachine.c:482,716,797
 *   cpb_split_points                             getSplitPoints                         impl/pairwiseAligner.c:1230
 *   cpb_band                                     band_construct / band_constructDynamic impl/pairwiseAligner.c:183,128
 *
 * There is no CPU fallback: every compute entry point needs a CUDA device and returns
 * CPB_ERR_CUDA (with a message from cpb_last_error) when none is usable.
 */
#ifndef CPECAN_B200_H_
#define CPECAN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CPB_PAIR_ALIGNMENT_PROB_1 10000000 /* inc/pairwiseAligner.h:26 */

enum {
    CPB_OK = 0,
    CPB_ERR_CUDA = 1,          /* no device / CUDA runtime failure */
    CPB_ERR_ARGUMENT = 2,      /* bad parameter (cf. the reference's asserts, impl/pairwiseAligner.c:761-765) */
    CPB_ERR_BAND = 3,          /* invalid diagonal (reference: PAIRWISE_ALIGNMENT_EXCEPTION, :31-35) */
    CPB_ERR_BAND_TOO_WIDE = 4, /* a band diagonal is wider than the widest kernel configuration */
    CPB_ERR_MEMORY = 5
};

/* StateMachineType, inc/stateMachine.h:28-33 */
enum { CPB_FIVE_STATE = 0, CPB_FIVE_STATE_ASYMMETRIC = 1, CPB_THREE_STATE = 2, CPB_THREE_STATE_ASYMMETRIC = 3 };

enum { CPB_MODE_ALIGNED_PAIRS = 0, CPB_MODE_ALIGNED_PAIRS_INDELS = 1, CPB_MODE_EXPECTATIONS = 2, CPB_MODE_FORWARD = 3 };

/* PairwiseAlignmentParameters, inc/pairwiseAligner.h:28-41 (same fields, same meaning, fixed-width types) */
typedef struct {
    double threshold;
    int64_t minDiagsBetweenTraceBack;
    int64_t traceBackDiagonals;
    int64_t diagonalExpansion;
    int64_t constraintDiagonalTrim;
    int64_t anchorMatrixBiggerThanThis;
    int64_t repeatMaskMatrixBiggerThanThis;
    int64_t splitMatrixBiggerThanThis;
    int32_t alignAmbiguityCharacters;
    float gapGamma;
    int32_t dynamicAnchorExpansion;
    int32_t pad_;
} CpbParams;

/*
 * Flat, vtable-free image of a StateMachine5 / StateMachine3 (impl/stateMachine.c:377-399, :631-646):
 * log-space transitions in the order the reference's cellCalculate issues them, per neighbour group,
 * and 5x5 / 5 emission tables that already contain the N rows (impl/stateMachine.c:351-366).
 *   five-state : lower  M->sGX, sGX->sGX, M->lGX, lGX->lGX
 *                middle M->M, sGX->M, sGY->M, lGX->M, lGY->M
 *                upper  M->sGY, sGY->sGY, M->lGY, lGY->lGY
 *   three-state: lower  M->gX, gX->gX, gY->gX;  middle M->M, gX->M, gY->M;  upper M->gY, gY->gY, gX->gY
 */
typedef struct {
    int32_t type;        /* CPB_FIVE_STATE ... */
    int32_t stateNumber; /* 5 or 3 */
    double start[5], raggedStart[5], end[5], raggedEnd[5];
    double tLower[4], tMiddle[5], tUpper[4];
    double eMatch[25]; /* [cX*5 + cY], cX,cY in a,c,g,t,n */
    double eGapX[5], eGapY[5];
} CpbModel;

/* Hmm expectation block (inc/stateMachine.h:61-67) flattened: transitions[S*S] row-major from*S+to,
 * emissions[S*16] state*16+x*4+y, then likelihood. */
#define CPB_HMM_LEN(S) ((S) * (S) + (S) * 16 + 1)

typedef struct cpb_context cpb_context;
typedef struct cpb_batch cpb_batch;

const char *cpb_version(void);
const char *cpb_last_error(void);

void cpb_params_default(CpbParams *p);
int cpb_model_default(int type, CpbModel *m);
/* transitions: S*S probabilities, emissions: S*16 probabilities (an Hmm as hmm_loadFromFile returns it) */
int cpb_model_from_hmm(int type, const double *transitions, const double *emissions, CpbModel *m);

/* Host-side helpers exposed for callers and for the reference's band / split-point unit tests.
 * anchors are (x, y, expansion) int64 triples, 0-based sequence coordinates. */
int64_t cpb_split_points(const int64_t *anchors, int64_t nAnchors, int64_t lX, int64_t lY, int64_t splitMatrixBiggerThanThis,
                         int raggedLeft, int raggedRight, int64_t *out4, int64_t cap);

/* ---- device context ---- */
/* stream: a cudaStream_t (as void*) the engine launches on, or NULL for the context's own stream. */
int cpb_context_create(int device, void *stream, cpb_context **out);
void cpb_context_destroy(cpb_context *ctx);
/* upper bound on scratch HBM per chunk (bytes); 0 = 70% of free memory at first use */
/* Page-locked host memory from the context's pool, for results the caller wants at the link's full rate (cpb_batch_fetch_* accept
 * any host pointer; into pageable memory the copy is several times slower).  NULL if it cannot be had.  Not thread safe per context. */
void *cpb_pinned_alloc(cpb_context *ctx, size_t bytes);
void cpb_pinned_free(cpb_context *ctx, void *p);
void cpb_context_set_scratch_budget(cpb_context *ctx, size_t bytes);

/* Device-side band builder for one region (what kernel K1 computes), copied back for inspection:
 * out3 receives (xay, xmyL, xmyR) for xay = 0..lX+lY.  Returns CPB_OK or CPB_ERR_BAND. */
int cpb_band(cpb_context *ctx, const int64_t *anchors, int64_t nAnchors, int64_t lX, int64_t lY, int64_t expansion, int dynamic,
             int64_t *out3);

/*
 * ---- batches ----
 * A batch is n independent alignment problems.  Sequences are given as one concatenated char buffer per
 * side plus n+1 offsets (any case, non-ACGT => N, no terminators needed); anchors as one int64 triple
 * array plus n+1 offsets (in triples); ragged flags per pair (may be NULL = all 0).
 * cpb_batch_create copies the inputs to the device (host pointers are not retained).
 */
int cpb_batch_create(cpb_context *ctx, int64_t nPairs, const char *seqX, const int64_t *xOff, const char *seqY, const int64_t *yOff,
                     const int64_t *anchors, const int64_t *anchorOff, const uint8_t *raggedLeft, const uint8_t *raggedRight,
                     cpb_batch **out);
/* As cpb_batch_create, with every pair's anchors found on the device: the triples, in order, that libcpecan.so's
 * getBlastPairsForPairwiseAlignmentParameters returns on the host.  Reads p->constraintDiagonalTrim, diagonalExpansion,
 * anchorMatrixBiggerThanThis, repeatMaskMatrixBiggerThanThis; cpb_batch_run takes its parameters as before.  Lower case is the soft
 * mask, as there.  The per-position work arrays are processed in chunks that fit the scratch budget; a single problem (a pair's
 * matrix, or a gap between its anchors) that does not fit returns CPB_ERR_MEMORY.  A negative trim or expansion, or an expansion of
 * 2^31 or more, returns CPB_ERR_ARGUMENT. */
int cpb_batch_create_anchored(cpb_context *ctx, int64_t nPairs, const char *seqX, const int64_t *xOff, const char *seqY,
                              const int64_t *yOff, const uint8_t *raggedLeft, const uint8_t *raggedRight, const CpbParams *p,
                              cpb_batch **out);
/* the anchors a batch holds, whoever made them: n+1 offsets (in triples), int64 (x, y, expansion) triples */
int64_t cpb_batch_anchor_count(const cpb_batch *b);
int cpb_batch_fetch_anchors(const cpb_batch *b, int64_t *offsets, int64_t *triples);
void cpb_batch_destroy(cpb_batch *b);

/* Runs the whole hot path on the device for the batch; results stay in HBM until fetched.
 * May be called repeatedly (e.g. for timing, or with a new model for the next EM iteration). */
int cpb_batch_run(cpb_batch *b, const CpbModel *m, const CpbParams *p, int mode);

typedef struct {
    int64_t nPairs, nRegions, nBlocks, nChunks;
    int64_t cells;         /* band cells, each counted once (SURVEY.md section 8d) */
    int64_t diagonals;     /* sum over regions of lX+lY+1 */
    int64_t outputTriples; /* total (p,x,y) triples produced (all lists) */
    int64_t kernelLaunches;
    double msBand, msForward, msBackward, msTotals, msPosterior; /* CUDA-event times of the last run, summed over chunks */
    int32_t maxWidth;
    int32_t twoPass;       /* 1 if the forward sweep ran as checkpoint pass + per-block recomputation (chunked runs of long regions) */
    double msCheckpoint;   /* part of msForward spent in the plane-less checkpoint pass (0 unless twoPass) */
    int64_t pintFixups;    /* weights floor(p * 1e7) the host recomputed with its own libm (cells within 2e-8 of an integer) */
    int64_t planReused;    /* 1 if this run kept the regions, bands, schedule, chunks and work lists of the batch's previous run (same mode,
                            * state count, banding parameters and scratch budget; $CPB_NO_PLAN_CACHE=1 turns that off) */
    int64_t reweighted;    /* 1 once cpb_batch_reweight_pairs has rewritten list 0 of this run: fetches and scores then see those weights */
} CpbRunStats;
/* Result sink: a host buffer (page-locked for full speed: cpb_pinned_alloc, cudaHostAlloc, torch pin_memory) of capacityTriples
 * (pInt, x, y) int32 triples that the next runs fill with list `list` WHILE they compute -- every chunk's triples are copied out on a
 * second stream beside the next chunk's kernels, so the device-to-host copy of the whole list (1.3 GB per 100 000 x 1 kb pairs)
 * is off the critical path.  cpb_batch_fetch_pairs called with that same pointer then only hands over the offsets.  If a run
 * produces more than the capacity the sink is skipped for that run and the fetch copies as usual.  NULL / 0 removes the sink. */
int cpb_batch_set_result_sink(cpb_batch *b, int list, int32_t *hostTriples, int64_t capacityTriples);

void cpb_batch_stats(const cpb_batch *b, CpbRunStats *out);

/* Results of the last run.  list: 0 = match, 1 = gapX, 2 = gapY (the latter two only in INDELS mode).
 * offsets receives n+1 entries (in triples); triples are int32 (pInt, x, y), 0-based sequence
 * coordinates, grouped by pair in input order; within a pair: region, block, diagonal (x+y) and x ascending. */
int64_t cpb_batch_result_count(const cpb_batch *b, int list);
int cpb_batch_fetch_pairs(cpb_batch *b, int list, int64_t *offsets, int32_t *triples);
/* As cpb_batch_fetch_pairs, with every pair's triples in the order the reference's own lists have (regions ascending; inside a region
 * the traceback blocks last to first; inside a block x+y ascending and x descending): what libcpecan.so returns, so that callers whose
 * result depends on list order (impl/pairwiseAligner.c:1603-1724) behave as with the reference. */
int cpb_batch_fetch_pairs_reference_order(cpb_batch *b, int list, int64_t *offsets, int32_t *triples);
/* Post-posterior filters on the device (list 0 of the last ALIGNED_PAIRS / ALIGNED_PAIRS_INDELS run; SURVEY.md section 8f, N2).
 * cpb_batch_reweight_pairs: every weight becomes weight - gapGamma * (gap weight of its x + gap weight of its y), where the gap
 * weight of a position is PAIR_ALIGNMENT_PROB_1 minus the weights aligned to it, floored at 0 -- reweightAlignedPairs2 of
 * impl/pairwiseAligner.c:1519-1560, in place, before the pairs are fetched; gapGamma <= 0 leaves them alone, as there.  Once per
 * run: CpbRunStats.reweighted says that list 0 now holds these weights, a second call is an error, cpb_batch_run resets it.
 * cpb_batch_alignment_scores: per pair, getAlignmentScore of impl/multipleAligner.c:604-619 (n int64 values to the host). */
int cpb_batch_reweight_pairs(cpb_batch *b, double gapGamma);
int cpb_batch_alignment_scores(cpb_batch *b, int64_t *scores);
/*
 * Decoders: one alignment per pair from the lists of the last run, on the device, into the batch's alignment list -- n+1 offsets and
 * int32 (pInt, x, y) triples, 0-based, like the result lists; per pair the pairs of the alignment, x and y strictly increasing.  Each
 * returns, at tolerance 0 (same triples, same order, same double bits), what the host function of libcpecan.so (host/realign.c) returns on
 * the lists libcpecan.so would hand it.  Each decode call replaces the alignment list; cpb_batch_run clears it; cpb_batch_reweight_pairs
 * does not touch it.  Work arrays are processed in chunks that fit the scratch budget; a single pair that does not fit returns
 * CPB_ERR_MEMORY.  libcpecan.so and cPecanRealign still decode on the host.
 *
 * cpb_batch_ordered_chain: filterPairwiseAlignmentToMakePairsOrdered (impl/multipleAligner.c:945-972; realign.c:150-247) of list 0 as it
 *   stands (reweighted if cpb_batch_reweight_pairs was called, as cPecanRealign does): the heaviest chain, strictly increasing in x and y,
 *   of the pairs with weight / PAIR_ALIGNMENT_PROB_1 >= matchGamma and > 0.  matchGamma in [0, 1].  Needs an ALIGNED_PAIRS or
 *   ALIGNED_PAIRS_INDELS run.
 * cpb_batch_mea: getMaximalExpectedAccuracyPairwiseAlignment (impl/pairwiseAligner.c:1603-1724; realign.c:249-326) of list 0 in the order
 *   cpb_batch_fetch_pairs_reference_order gives, with lists 1 and 2 as the gap weights and gapGamma >= 0 as p->gapGamma; with leftShift
 *   set, followed by leftShiftAlignment (:1726-1767; realign.c:330-356), which is getShiftedMEAAlignment (:1769-1792).  scores (n doubles,
 *   or NULL) receives every pair's alignmentScore.  Needs an ALIGNED_PAIRS_INDELS run.
 * cpb_batch_score_alignments: per pair, scoreByIdentity, scoreByIdentityIgnoringGaps, scoreByPosteriorProbability or
 *   scoreByPosteriorProbabilityIgnoringGaps (impl/pairwiseAligner.c:1562-1597; realign.c:113-148) of its alignment; the two "ignoring
 *   gaps" forms are NaN for an empty alignment, as on the host.  Letters compare case-blind, N never matches.
 * Fetching or scoring before a decode call, a decode after an EXPECTATIONS or FORWARD run, and gammas or kind out of range return
 * CPB_ERR_ARGUMENT.  A decode call that returns an error, for whatever reason, leaves no alignment list (the previous one is gone too).
 * cpb_batch_alignments_count is 0 while there is no alignment list.
 */
enum { CPB_SCORE_IDENTITY = 0, CPB_SCORE_IDENTITY_IGNORING_GAPS = 1, CPB_SCORE_POSTERIOR = 2, CPB_SCORE_POSTERIOR_IGNORING_GAPS = 3 };
int cpb_batch_ordered_chain(cpb_batch *b, float matchGamma);
int cpb_batch_mea(cpb_batch *b, float gapGamma, int leftShift, double *scores);
int64_t cpb_batch_alignments_count(const cpb_batch *b);
int cpb_batch_fetch_alignments(const cpb_batch *b, int64_t *offsets, int32_t *triples);
int cpb_batch_score_alignments(cpb_batch *b, int kind, double *scores);
/*
 * Re-anchoring from the alignment list, for the next run of the same batch (cPecanEm --updateTheBand): replaces every pair's anchors with
 * those its alignment gives (p->constraintDiagonalTrim, p->diagonalExpansion) -- exactly the triples cPecanRealign's job_prepare
 * (host/realignJobs.h) builds from the cigar cPecanRealign writes for that alignment.  The alignment's maximal diagonal runs are the cigar's
 * match operations; a run of length L gives its columns at positions [trim, L - trim) (convertPairwiseForwardStrandAlignmentToAnchorPairs,
 * mismatched columns counted); each becomes (x, y, diagonalExpansion) and is kept iff its two bytes are equal after toupper and not N.
 * Per pair x ascending.  Needs an alignment list (cpb_batch_ordered_chain or cpb_batch_mea); without one, with p NULL, or with a trim or
 * expansion outside [0, 2^31) it returns CPB_ERR_ARGUMENT.  All or nothing: on any error, CPB_ERR_MEMORY for a pair whose work array does
 * not fit the scratch budget included, the batch keeps its anchors.  On success cpb_batch_anchor_count / cpb_batch_fetch_anchors return the
 * new anchors and the next cpb_batch_run plans anew (planReused 0); the lists of the last run, the alignment list and its scores stay as
 * they were.  The batch then runs as one cpb_batch_create makes from the fetched anchors.
 */
int cpb_batch_anchors_from_alignments(cpb_batch *b, const CpbParams *p);
/* device pointers of the same (valid until the next run / destroy) */
const int32_t *cpb_batch_device_triples(const cpb_batch *b, int list);
/* EXPECTATIONS mode: perPair (may be NULL) receives n * CPB_HMM_LEN(S) doubles, total receives CPB_HMM_LEN(S) doubles
 * (the sum over pairs, in pair order). */
int cpb_batch_fetch_expectations(cpb_batch *b, double *perPair, double *total);
const double *cpb_batch_device_expectation_total(const cpb_batch *b);
/* EM over several GPUs of one process: replaces every batch's device-resident expectation total by the sum over all n batches (one
 * per device, all from expectation-mode runs with the same model) with one ncclAllReduce(ncclDouble, ncclSum) per device
 * (cPecanEm.py:182-188 sums expectation files).  NCCL is loaded at run time; CPB_ERR_CUDA with a message if it is not there, and the
 * caller may then sum the per-batch totals itself. */
int cpb_expectations_allreduce(cpb_batch *const *batches, int n);

/* FORWARD mode: n log-probabilities */
int cpb_batch_fetch_forward(cpb_batch *b, double *logProb);

#ifdef __cplusplus
}
#endif
#endif /* CPECAN_B200_H_ */
