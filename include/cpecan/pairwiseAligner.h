/*
 * cpecan/pairwiseAligner.h -- cPecan's pairwise pair-HMM API (inc/pairwiseAligner.h of the reference) served by
 * libcpecan.so: plain C host code over the batched CUDA engine of include/cpecan_b200.h.
 *
 * Every function below keeps the reference's name, argument order, ownership rules and error convention
 * (st_errAbort on unusable input; a missing or failing CUDA device is reported the same way -- there is no host
 * implementation of the DP to fall back to).  Citations are to the reference tree.
 *
 * New in this library (the reference handles one pair per call): the *Batch entry points at the end, which run
 * many independent pairs in one device pass and are what cPecanRealign's per-cigar loop (cPecanRealign.c:509-605)
 * and multipleAligner's all-pairs loop (impl/multipleAligner.c:668-681) should call.
 */
#ifndef CPECAN_PAIRWISEALIGNER_H_
#define CPECAN_PAIRWISEALIGNER_H_

#include "cpecan/sonLibLite.h"
#include "cpecan/stateMachine.h"

#ifdef __cplusplus
extern "C" {
#endif

extern const char *PAIRWISE_ALIGNMENT_EXCEPTION_ID; /* inc/pairwiseAligner.h:23 */

#define PAIR_ALIGNMENT_PROB_1 10000000 /* inc/pairwiseAligner.h:26 */
#define LOG_ZERO (-INFINITY)           /* inc/pairwiseAligner.h:165 */
#define LOG_ONE 0.0

/* inc/pairwiseAligner.h:28-41, same fields in the same order */
typedef struct _pairwiseAlignmentBandingParameters {
    double threshold;
    int64_t minDiagsBetweenTraceBack;
    int64_t traceBackDiagonals;
    int64_t diagonalExpansion;
    int64_t constraintDiagonalTrim;
    int64_t anchorMatrixBiggerThanThis;
    int64_t repeatMaskMatrixBiggerThanThis;
    int64_t splitMatrixBiggerThanThis;
    bool alignAmbiguityCharacters;
    float gapGamma;
    bool dynamicAnchorExpansion;
} PairwiseAlignmentParameters;

PairwiseAlignmentParameters *pairwiseAlignmentBandingParameters_construct(void);      /* :43, defaults of impl/pairwiseAligner.c:1334-1348 */
void pairwiseAlignmentBandingParameters_destruct(PairwiseAlignmentParameters *p);     /* :45 */
PairwiseAlignmentParameters *pairwiseAlignmentParameters_jsonParse(char *buf, size_t r); /* :51 */

/* :56 -- log P(x, y) by the banded forward algorithm */
double computeForwardProbability(char *seqX, char *seqY, stList *anchorPairs, PairwiseAlignmentParameters *p, StateMachine *sM,
                                 bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd);

/*
 * :62 / :69 -- as the ...UsingAnchors forms with anchors from getBlastPairsForPairwiseAlignmentParameters (below): matrices up
 * to p->anchorMatrixBiggerThanThis are aligned unanchored exactly as the reference does; larger ones are anchored in process
 * (the reference shells out to LASTZ here, impl/pairwiseAligner.c:1005-1080), or by the provider registered with
 * cpecan_setAnchorProvider if there is one.
 */
stList *getAlignedPairs(StateMachine *sM, const char *string1, const char *string2, PairwiseAlignmentParameters *p,
                        bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd);
void getAlignedPairsWithIndels(StateMachine *sM, const char *string1, const char *string2, PairwiseAlignmentParameters *p,
                               stList **alignedPairs, stList **gapXPairs, stList **gapYPairs, bool alignmentHasRaggedLeftEnd,
                               bool alignmentHasRaggedRightEnd);

/* :75 -- list of stIntTuple (pInt, x, y), 0-based, unique (x, y), caller frees with stList_destruct */
stList *getAlignedPairsUsingAnchors(StateMachine *sM, const char *sX, const char *sY, stList *anchorPairs, PairwiseAlignmentParameters *p,
                                    bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd);
/* :77 */
void getAlignedPairsWithIndelsUsingAnchors(StateMachine *sM, const char *sX, const char *sY, stList *anchorPairs,
                                           PairwiseAlignmentParameters *p, stList **alignedPairs, stList **gapXPairs, stList **gapYPairs,
                                           bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd);
/* :105 / :108 -- expected transition / emission counts are added to hmmExpectations */
void getExpectationsUsingAnchors(StateMachine *sM, Hmm *hmmExpectations, const char *sX, const char *sY, stList *anchorPairs,
                                 PairwiseAlignmentParameters *p, bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd);
void getExpectations(StateMachine *sM, Hmm *hmmExpectations, const char *sX, const char *sY, PairwiseAlignmentParameters *p,
                     bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd);

/* ---- helpers the reference exposes for its tests ---- */

/* :116-138 */
typedef struct _diagonal {
    int64_t xay;  /* x + y */
    int64_t xmyL; /* smallest x - y */
    int64_t xmyR; /* largest x - y */
} Diagonal;

Diagonal diagonal_construct(int64_t xay, int64_t xmyL, int64_t xmyR); /* aborts on an invalid diagonal (reference: stThrowNew) */
int64_t diagonal_getXay(Diagonal diagonal);
int64_t diagonal_getMinXmy(Diagonal diagonal);
int64_t diagonal_getMaxXmy(Diagonal diagonal);
int64_t diagonal_getWidth(Diagonal diagonal);
int64_t diagonal_getXCoordinate(int64_t xay, int64_t xmy);
int64_t diagonal_getYCoordinate(int64_t xay, int64_t xmy);
int64_t diagonal_equals(Diagonal diagonal1, Diagonal diagonal2);

/* :140-161 -- the band comes from the device-side band builder (kernel k_band) */
typedef struct _band Band;
typedef struct _bandIterator BandIterator;
Band *band_construct(stList *anchorPairs, int64_t lX, int64_t lY, int64_t expansion);
Band *band_constructDynamic(stList *anchorPairs, int64_t lX, int64_t lY);
void band_destruct(Band *band);
BandIterator *bandIterator_construct(Band *band);
void bandIterator_destruct(BandIterator *bandIterator);
BandIterator *bandIterator_clone(BandIterator *bandIterator);
Diagonal bandIterator_getNext(BandIterator *bandIterator);
Diagonal bandIterator_getPrevious(BandIterator *bandIterator);

/* :171-175 */
Symbol symbol_convertCharToSymbol(char i);
char symbol_convertSymbolToChar(Symbol i);
Symbol *symbol_convertStringToSymbols(const char *s, int64_t sL);

/* :167 -- the reference's log-space addition: 4-segment cubic with float-literal coefficients, cut-off at 7.5
 * (impl/pairwiseAligner.c:287-307).  A scalar helper for callers and tests; the device kernels carry their own copy. */
double logAdd(double x, double y);

/* :177-182 */
typedef struct _symbolString {
    Symbol *sequence;
    int64_t length;
} SymbolString;
SymbolString symbolString_construct(const char *sequence, int64_t length);
void symbolString_destruct(SymbolString s);

/*
 * :233-247, :264 -- the banded forward-backward itself, with the per-diagonal posterior callback the reference passes in.
 *
 * On the device the per-diagonal work is compiled into the kernels, so a callback cannot cross: the three callbacks the
 * reference's own wrappers use (impl/pairwiseAligner.c:1441, :1472, :1502) are exported under their names and recognised BY
 * ADDRESS -- diagonalCalculationPosteriorMatchProbs selects the aligned-pairs mode (extraArgs[0] = list of (pInt, x, y)),
 * diagonalCalculationPosteriorProbs the match + gap-X + gap-Y mode (extraArgs[0], [2], [4]), diagonalCalculationExpectations
 * the expectation mode (extraArgs = Hmm *, +=).  Any other function pointer aborts with a message, and so does calling one of
 * the three directly (DpMatrix is never materialised on the host).  Lists are filled in the reference's own emission order
 * (traceback blocks ascending, diagonals descending, x ascending) with coordinates relative to the strings passed in.
 */
typedef struct _dpMatrix DpMatrix;
typedef void (*DiagonalPosteriorProbFn)(StateMachine *, int64_t, DpMatrix *, DpMatrix *, const SymbolString, const SymbolString, double,
                                        PairwiseAlignmentParameters *, void *);
void diagonalCalculationPosteriorMatchProbs(StateMachine *sM, int64_t xay, DpMatrix *forwardDpMatrix, DpMatrix *backwardDpMatrix,
                                            const SymbolString sX, const SymbolString sY, double totalProbability,
                                            PairwiseAlignmentParameters *p, void *extraArgs); /* :233 */
void diagonalCalculationPosteriorProbs(StateMachine *sM, int64_t xay, DpMatrix *forwardDpMatrix, DpMatrix *backwardDpMatrix,
                                       const SymbolString sX, const SymbolString sY, double totalProbability,
                                       PairwiseAlignmentParameters *p, void *extraArgs); /* impl/pairwiseAligner.c:691 */
void diagonalCalculationExpectations(StateMachine *sM, int64_t xay, DpMatrix *forwardDpMatrix, DpMatrix *backwardDpMatrix,
                                     const SymbolString sX, const SymbolString sY, double totalProbability,
                                     PairwiseAlignmentParameters *p, void *extraArgs); /* impl/pairwiseAligner.c:735 (static there) */
/* :245 -- one region, no splitting */
void getPosteriorProbsWithBanding(StateMachine *sM, stList *anchorPairs, const SymbolString sX, const SymbolString sY,
                                  PairwiseAlignmentParameters *p, bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd,
                                  DiagonalPosteriorProbFn diagonalPosteriorProbFn, void *extraArgs);
/* :264 -- splits at anchor gaps bigger than p->splitMatrixBiggerThanThis; after every region (all of them computed in one
 * device pass) its results are appended and coordinateCorrectionFn(x1, y1, extraArgs) is called, if not NULL */
void getPosteriorProbsWithBandingSplittingAlignmentsByLargeGaps(StateMachine *sM, stList *anchorPairs, const char *sX, const char *sY, int64_t lX,
                                                                int64_t lY, PairwiseAlignmentParameters *p, bool alignmentHasRaggedLeftEnd,
                                                                bool alignmentHasRaggedRightEnd, DiagonalPosteriorProbFn diagonalPosteriorProbFn,
                                                                void (*coordinateCorrectionFn)(), void *extraArgs);

/* :251-257 -- anchors found in process by a seed-and-chain aligner (host/anchors.c) where the reference shells out to LASTZ; same
 * contract: (x, y, diagonalExpansion) tuples sorted by x + y, every match run given column by column with `trim` columns dropped at
 * both ends; repeatMask: lower-case bases do not seed.  filterToRemoveOverlap and the two-level scheme are the reference's own. */
stList *getBlastPairs(const char *sX, const char *sY, int64_t lX, int64_t lY, int64_t trim, int64_t diagonalExpansion, bool repeatMask);
stList *getBlastPairsForPairwiseAlignmentParameters(const char *sX, const char *sY, const int64_t lX, const int64_t lY, PairwiseAlignmentParameters *p);
stList *filterToRemoveOverlap(stList *overlappingPairs);

/* :261 -- list of stIntTuple (x1, y1, x2, y2) */
stList *getSplitPoints(stList *anchorPairs, int64_t lX, int64_t lY, int64_t maxMatrixSize, bool alignmentHasRaggedLeftEnd,
                       bool alignmentHasRaggedRightEnd);

/* ---- after the device pass: host-side list work on the compacted output (cpecan_b200/csrc/host/realign.c) ---- */

struct PairwiseAlignment; /* cpecan/pairwiseAlignment.h */

/* :73 -- (x, y, diagonalExpansion) for every column of every match run of a forward-strand cigar, `trim` columns dropped at both ends */
stList *convertPairwiseForwardStrandAlignmentToAnchorPairs(struct PairwiseAlignment *pA, int64_t trim, int64_t diagonalExpansion);
/* :85-99 -- maximal expected accuracy subset of alignedPairs, its left shift, and both after an alignment */
stList *getMaximalExpectedAccuracyPairwiseAlignment(stList *alignedPairs, stList *gapXPairs, stList *gapYPairs, int64_t seqXLength,
                                                    int64_t seqYLength, double *alignmentScore, PairwiseAlignmentParameters *p);
stList *leftShiftAlignment(stList *alignedPairs, char *seqX, char *seqY);
stList *getShiftedMEAAlignment(char *seqX, char *seqY, stList *anchorAlignment, PairwiseAlignmentParameters *p, StateMachine *sM,
                               bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd, double *alignmentScore);
/* :272-278 -- probability of each position being aligned to a gap, and weights reduced by gapGamma times it (consumes alignedPairs) */
int64_t *getIndelProbabilities(stList *alignedPairs, int64_t seqLength, bool xIfTrueElseY);
stList *reweightAlignedPairs(stList *alignedPairs, int64_t *indelProbsX, int64_t *indelProbsY, double gapGamma);
stList *reweightAlignedPairs2(stList *alignedPairs, int64_t seqLengthX, int64_t seqLengthY, double gapGamma);
/* :287-307 */
int64_t getNumberOfMatchingAlignedPairs(char *subSeqX, char *subSeqY, stList *alignedPairs);
double scoreByIdentity(char *subSeqX, char *subSeqY, int64_t lX, int64_t lY, stList *alignedPairs);
double scoreByIdentityIgnoringGaps(char *subSeqX, char *subSeqY, stList *alignedPairs);
double scoreByPosteriorProbability(int64_t lX, int64_t lY, stList *alignedPairs);
double scoreByPosteriorProbabilityIgnoringGaps(stList *alignedPairs);

/* ---- batched entry points (not in the reference) ---- */

/* Anchor provider used by getAlignedPairs / getAlignedPairsWithIndels / getExpectations for matrices bigger than
 * p->anchorMatrixBiggerThanThis: returns a new stList of stIntTuple (x, y, expansion), strictly increasing in x and y. */
typedef stList *(*CpecanAnchorProvider)(const char *sX, const char *sY, int64_t lX, int64_t lY, PairwiseAlignmentParameters *p, void *extra);
void cpecan_setAnchorProvider(CpecanAnchorProvider provider, void *extra);

/* CUDA device used by this process (default: $CPECAN_DEVICE or 0).  Must be called before the first alignment. */
void cpecan_setDevice(int device);
/* The first n CUDA devices of the box (default: $CPECAN_DEVICES, else one device): every *Batch call and every resident batch then
 * deals its problems over the n GPUs -- longest first, by estimated band cells -- with one host thread, context and stream per GPU and
 * the results back at the problems' own indices; expectation totals are summed across the GPUs with one NCCL all-reduce. */
void cpecan_setDevices(int n);
/* the same with explicit device ordinals ($CPECAN_DEVICE_LIST="0,2,3") */
void cpecan_setDeviceList(const int *devices, int n);
int cpecan_getDeviceCount(void);
/* releases the device context (optional; also safe to never call) */
void cpecan_shutdown(void);

/* n independent problems in one device pass.  anchorPairs[i] may be NULL (no anchors); raggedLeft / raggedRight may
 * be NULL (all false).  Returns a new array of n lists (free each with stList_destruct, the array with free). */
stList **getAlignedPairsUsingAnchorsBatch(StateMachine *sM, int64_t n, const char *const *sX, const char *const *sY,
                                          stList *const *anchorPairs, PairwiseAlignmentParameters *p, const bool *raggedLeft,
                                          const bool *raggedRight);
/* the same from raw sequences: every problem is anchored as getAlignedPairs does (on the host threads), then all run in one device pass */
stList **getAlignedPairsBatch(StateMachine *sM, int64_t n, const char *const *sX, const char *const *sY, PairwiseAlignmentParameters *p,
                              const bool *raggedLeft, const bool *raggedRight);
/* the same followed by reweightAlignedPairs2(pairs, lX, lY, gapGamma) (:278) for every problem, done on the device before the
 * pairs come back (SURVEY.md section 8f, N2) */
stList **getReweightedAlignedPairsUsingAnchorsBatch(StateMachine *sM, int64_t n, const char *const *sX, const char *const *sY,
                                                    stList *const *anchorPairs, PairwiseAlignmentParameters *p, const bool *raggedLeft,
                                                    const bool *raggedRight, double gapGamma);
void getAlignedPairsWithIndelsUsingAnchorsBatch(StateMachine *sM, int64_t n, const char *const *sX, const char *const *sY,
                                                stList *const *anchorPairs, PairwiseAlignmentParameters *p, stList ***alignedPairs,
                                                stList ***gapXPairs, stList ***gapYPairs, const bool *raggedLeft, const bool *raggedRight);
/* sums the expectations of all n problems into hmmExpectations (+=), as n calls of getExpectationsUsingAnchors would */
void getExpectationsUsingAnchorsBatch(StateMachine *sM, Hmm *hmmExpectations, int64_t n, const char *const *sX, const char *const *sY,
                                      stList *const *anchorPairs, PairwiseAlignmentParameters *p, const bool *raggedLeft,
                                      const bool *raggedRight);
void computeForwardProbabilityBatch(StateMachine *sM, int64_t n, const char *const *sX, const char *const *sY, stList *const *anchorPairs,
                                    PairwiseAlignmentParameters *p, const bool *raggedLeft, const bool *raggedRight, double *logProbs);

/* A batch whose sequences and anchors stay on the device: EM runs the expectation pass over the same alignments once per iteration
 * with a new model (cPecanEm.py:176-215 re-reads everything through a cPecanRealign subprocess per iteration and alignment file). */
typedef struct _cpecanResidentBatch CpecanResidentBatch;
CpecanResidentBatch *cpecanResidentBatch_construct(int64_t n, const char *const *sX, const char *const *sY, stList *const *anchorPairs,
                                                   PairwiseAlignmentParameters *p, const bool *raggedLeft, const bool *raggedRight);
void cpecanResidentBatch_destruct(CpecanResidentBatch *batch);
/* += into hmmExpectations, as getExpectationsUsingAnchorsBatch */
void cpecanResidentBatch_getExpectations(CpecanResidentBatch *batch, StateMachine *sM, Hmm *hmmExpectations, PairwiseAlignmentParameters *p);
/* Re-anchors every alignment of the batch under sM, on every device (one host thread each), with no list leaving the device: an
 * ALIGNED_PAIRS run with p, reweighting by p->gapGamma, the heaviest ordered chain at matchGamma, then the anchors of that chain as
 * cPecanRealign's cigar would give them (p->constraintDiagonalTrim, p->diagonalExpansion; cpb_batch_anchors_from_alignments).  These are
 * cPecanRealign's default steps; the next expectation pass runs in the new band.  An invalid band aborts with
 * PAIRWISE_ALIGNMENT_EXCEPTION, any other engine error as cpecanResidentBatch_getExpectations does. */
void cpecanResidentBatch_updateAnchors(CpecanResidentBatch *batch, StateMachine *sM, PairwiseAlignmentParameters *p, float matchGamma);

#ifdef __cplusplus
}
#endif
#endif /* CPECAN_PAIRWISEALIGNER_H_ */
