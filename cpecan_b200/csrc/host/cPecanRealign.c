/*
 * cPecanRealign -- realigns pairwise alignments (cigars on stdin) with the pair-HMM and writes them back (stdout), or
 * accumulates EM expectations over them.  Same command line, file formats and per-alignment processing as the reference's
 * cPecanRealign.c (options :374-473, coordinate handling :509-523, post-processing :546-599, expectations :530-535 and :608-614).
 *
 * What is different is the shape of the loop.  The reference runs one alignment at a time through the CPU DP
 * (cPecanRealign.c:509-605).  Here the cigars are read in batches and every batch goes through ONE device pass of libcpecan.so:
 * getRealignedCigarsUsingAnchorsBatch runs the pair-HMM, reweights, chains, scores and builds the output's cigar operations on the
 * device, so only operations and scores (and, for the posterior files, triples) come back; --rescoreOriginalAlignment takes the
 * posteriors (getAlignedPairsUsingAnchorsBatch) and --outputExpectations the expectations (getExpectationsUsingAnchorsBatch).  The
 * host threads prepare the sub-sequences and anchors before the pass and write the cigars after it; output order is input order.
 * There is no host DP: without a CUDA device the program aborts with the engine's message.
 */
#include <getopt.h>
#include <time.h>

#include "cpecan/multipleAligner.h"
#include "host_internal.h"
#include "realignJobs.h"

static void usage(void) {
    fprintf(stderr, "cPecanRelign [options] seq1[fasta] seq2[fasta], version 0.2 (B200 batched engine)\n");
    fprintf(stderr, "Realigns a set of pairwise alignments, as cigars, read from the command line and written back to the command line\n");
    fprintf(stderr, "-a --logLevel : Set the log level\n");
    fprintf(stderr, "-l --gapGamma : (float >= 0) The gap gamma (as in the AMAP function)\n");
    fprintf(stderr, "-L --matchGamma : (float [0, 1]) The match gamma (the avg. weight or greater to be allowed in the alignment)\n");
    fprintf(stderr, "-o --splitMatrixBiggerThanThis : (int >= 0)  No dp matrix bigger than this number squared will be computed.\n");
    fprintf(stderr, "-r --diagonalExpansion : (int >= 0 and even) Number of x-y diagonals to expand around anchors\n");
    fprintf(stderr, "-t --constraintDiagonalTrim : (int >= 0) Amount to trim from ends of each anchor\n");
    fprintf(stderr, "-w --alignAmbiguityCharacters : Align ambiguity characters (anything not ACTGactg) as a wildcard\n");
    fprintf(stderr, "-x --rescoreOriginalAlignment : Rescore the original alignment. The output cigar is the same alignment.\n");
    fprintf(stderr, "-i --rescoreByIdentity : Set score equal to alignment identity, treating indels as mismatches.\n");
    fprintf(stderr, "-j --rescoreByPosteriorProb : Set score equal to avg. posterior match probability, treating indels as residues with 0 match probability.\n");
    fprintf(stderr, "-k --rescoreByIdentityIgnoringGaps : Set score equal to alignment identity, ignoring indels.\n");
    fprintf(stderr, "-m --rescoreByPosteriorProbIgnoringGaps : Set score equal to avg. posterior match probability, ignoring gaps.\n");
    fprintf(stderr, "-h --help : Print this help screen\n");
    fprintf(stderr, "-s --splitIndelsLongerThanThis : Split alignments with consecutive runs of indels that are longer than this.\n");
    fprintf(stderr, "-u --outputPosteriorProbs [FILE] : Outputs the posterior match probs of positions in the alignment to the given tab separated file, each line being X-coordinate, Y-coordinate, posterior-match prob.\n");
    fprintf(stderr, "-z --outputAllPosteriorProbs [FILE] : As --outputPosteriorProbs, but for all pairs in the banded alignment\n");
    fprintf(stderr, "-v --outputExpectations [FILE] : Instead of realigning, switches to calculating expectations, dumping out expectations as matrix in the given file.\n");
    fprintf(stderr, "-y --loadHmm [FILE] : Loads HMM from given file.\n");
    fprintf(stderr, "-b --batchBases : (int > 0) Bases of sequence per device pass (default 200000000; not in the reference)\n");
    fprintf(stderr, "--gpus N : spread every device pass over the first N GPUs of the box (default $CPECAN_DEVICES or 1; not in the reference)\n");
}

static int64_t transform_coordinate(int64_t c, int64_t shift, bool flip, int64_t seqLength) { return shift + (flip ? seqLength - 1 - c : c); }

/* n (pInt, x, y) triples, in original coordinates */
static void write_posterior_probs(const char *file, const int32_t *pairs, int64_t n, const Job *j) {
    const struct PairwiseAlignment *pA = j->pA;
    FILE *f = fopen(file, "w");
    if (f == NULL) st_errAbort("cPecanRealign: cannot write %s", file);
    for (int64_t i = 0; i < n; i++) {
        fprintf(f, "%" PRIi64 "\t%" PRIi64 "\t%f\n", transform_coordinate(pairs[3 * i + 1], j->shift1, j->flip1, pA->end1 - pA->start1),
                transform_coordinate(pairs[3 * i + 2], j->shift2, j->flip2, pA->end2 - pA->start2), ((double) pairs[3 * i]) / PAIR_ALIGNMENT_PROB_1);
    }
    fclose(f);
}

static void write_posterior_list(const char *file, stList *pairs, const Job *j) {
    const int64_t n = stList_length(pairs);
    int32_t *t = xmalloc((size_t) n * 3 * sizeof(int32_t));
    for (int64_t i = 0; i < n; i++) {
        for (int64_t k = 0; k < 3; k++) t[3 * i + k] = (int32_t) stIntTuple_get(stList_get(pairs, i), k);
    }
    write_posterior_probs(file, t, n, j);
    free(t);
}

/* ---- the original alignment's columns with their posterior weights (cPecanRealign.c:322-353) ---- */

static int by_xy(const void *a, const void *b) {
    const int64_t *p = a, *q = b;
    if (p[0] != q[0]) return p[0] < q[0] ? -1 : 1;
    return p[1] < q[1] ? -1 : (p[1] > q[1] ? 1 : 0);
}

static stList *score_anchor_pairs(stList *anchorPairs, stList *alignedPairs) {
    const int64_t n = stList_length(anchorPairs);
    int64_t *a = xmalloc((size_t) n * 3 * sizeof(int64_t)); /* (x, y, weight or -1 = not seen) */
    for (int64_t i = 0; i < n; i++) {
        stIntTuple *t = stList_get(anchorPairs, i);
        a[3 * i] = stIntTuple_get(t, 0);
        a[3 * i + 1] = stIntTuple_get(t, 1);
        a[3 * i + 2] = -1;
    }
    qsort(a, (size_t) n, 3 * sizeof(int64_t), by_xy);
    stList *scored = stList_construct3(0, (void (*)(void *)) stIntTuple_destruct);
    for (int64_t i = 0; i < stList_length(alignedPairs); i++) {
        stIntTuple *t = stList_get(alignedPairs, i);
        int64_t key[3] = { stIntTuple_get(t, 1), stIntTuple_get(t, 2), 0 };
        int64_t *hit = bsearch(key, a, (size_t) n, 3 * sizeof(int64_t), by_xy);
        if (hit != NULL && hit[2] < 0) {
            hit[2] = stIntTuple_get(t, 0);
            stList_append(scored, stIntTuple_construct3(hit[2], hit[0], hit[1]));
        }
    }
    /* columns of the original alignment below the posterior threshold get weight 0 */
    for (int64_t i = 0; i < n; i++) {
        if (a[3 * i + 2] < 0) stList_append(scored, stIntTuple_construct3(0, a[3 * i], a[3 * i + 1]));
    }
    free(a);
    return scored;
}

/* ---- aligned pairs -> cigar (cPecanRealign.c:50-92), for --rescoreOriginalAlignment; the realignment's cigars come from the device ---- */

static void add_op(struct List *ops, int64_t type, int64_t length) { listAppend(ops, constructAlignmentOperation(type, length, 0)); }

/* xy: n (x, y) pairs sorted ascending */
static struct PairwiseAlignment *pairs_to_alignment(const char *name1, const char *name2, double score, int64_t length1, int64_t length2,
                                                    const int64_t *xy, int64_t n) {
    struct List *ops = constructEmptyList(0, (void (*)(void *)) destructAlignmentOperation);
    int64_t pX = -1, pY = -1, run = 0;
    for (int64_t i = 0; i <= n; i++) { /* a closing pair at (length1, length2) produces the trailing indels */
        const int64_t x = i < n ? xy[2 * i] : length1;
        const int64_t y = i < n ? xy[2 * i + 1] : length2;
        if (x - pX > 0 && y - pY > 0) { /* pairs that do not advance both sequences are dropped */
            if (x - pX > 1) {
                if (run > 0) add_op(ops, PAIRWISE_MATCH, run);
                run = 0;
                add_op(ops, PAIRWISE_INDEL_X, x - pX - 1);
            }
            if (y - pY > 1) {
                if (run > 0) add_op(ops, PAIRWISE_MATCH, run);
                run = 0;
                add_op(ops, PAIRWISE_INDEL_Y, y - pY - 1);
            }
            run++;
            pX = x;
            pY = y;
        }
    }
    if (run > 1) add_op(ops, PAIRWISE_MATCH, run - 1); /* the closing pair itself is not a column */
    return constructPairwiseAlignment(name1, 0, length1, 1, name2, 0, length2, 1, score, ops);
}

static int by_x_then_y(const void *a, const void *b) {
    const int64_t *p = a, *q = b;
    if (p[0] != q[0]) return p[0] < q[0] ? -1 : 1;
    return p[1] < q[1] ? -1 : (p[1] > q[1] ? 1 : 0);
}

/* ---- splitting at long indel runs (cPecanRealign.c:94-218) ---- */

static void flush_piece(stList *pieces, const struct PairwiseAlignment *pA, struct List **ops, int64_t start1, int64_t end1, int64_t start2, int64_t end2) {
    if ((*ops)->length != 0) {
        stList_append(pieces, constructPairwiseAlignment(pA->contig1, start1, end1, pA->strand1, pA->contig2, start2, end2, pA->strand2, pA->score, *ops));
    } else {
        destructList(*ops);
    }
    *ops = constructEmptyList(0, (void (*)(void *)) destructAlignmentOperation);
}

static stList *split_alignment(const struct PairwiseAlignment *pA, int64_t maxIndelLength) {
    stList *pieces = stList_construct3(0, (void (*)(void *)) destructPairwiseAlignment);
    struct List *ops = constructEmptyList(0, (void (*)(void *)) destructAlignmentOperation);
    struct List *pending = constructEmptyList(0, NULL); /* the indel run since the last match: kept only if a match follows */
    int64_t pos1 = pA->start1, pos2 = pA->start2, start1 = pos1, start2 = pos2, end1 = 0, end2 = 0, indelRun = 0;
    const int64_t step1 = pA->strand1 ? 1 : -1, step2 = pA->strand2 ? 1 : -1;
    for (int64_t i = 0; i < pA->operationList->length; i++) {
        const struct AlignmentOperation *op = pA->operationList->list[i];
        if (op->opType == PAIRWISE_MATCH) {
            if ((indelRun > maxIndelLength && ops->length != 0) || ops->length == 0) {
                /* an over-long run ends the piece before it; a run at the very start is dropped as well */
                if (ops->length != 0) flush_piece(pieces, pA, &ops, start1, end1, start2, end2);
                for (int64_t j = 0; j < pending->length; j++) destructAlignmentOperation(pending->list[j]);
                pending->length = 0;
                start1 = end1 = pos1;
                start2 = end2 = pos2;
            }
            indelRun = 0;
            for (int64_t j = 0; j < pending->length; j++) listAppend(ops, pending->list[j]);
            pending->length = 0;
            pos1 += step1 * op->length;
            pos2 += step2 * op->length;
            end1 = pos1;
            end2 = pos2;
            listAppend(ops, constructAlignmentOperation(op->opType, op->length, op->score));
        } else {
            indelRun += op->length;
            if (op->opType == PAIRWISE_INDEL_X) pos1 += step1 * op->length;
            else pos2 += step2 * op->length;
            listAppend(pending, constructAlignmentOperation(op->opType, op->length, op->score));
        }
    }
    flush_piece(pieces, pA, &ops, start1, end1, start2, end2);
    destructList(ops);
    for (int64_t j = 0; j < pending->length; j++) destructAlignmentOperation(pending->list[j]);
    destructList(pending);
    for (int64_t i = 0; i < stList_length(pieces); i++) checkPairwiseAlignment(stList_get(pieces, i));
    return pieces;
}

typedef struct {
    float matchGamma;
    bool rescoreOriginalAlignment, rescoreByIdentity, rescoreByPosteriorProbability, rescoreByIdentityIgnoringGaps,
        rescoreByPosteriorProbabilityIgnoringGaps;
    int64_t splitIndelsLongerThanThis; /* -1 = never */
    const char *posteriorProbsFile, *allPosteriorProbsFile;
} Options;

/* the score the options ask for (cPecanRealign.c:561-569: the first of these that is set), or -1 to keep the input's */
static int score_kind(const Options *o) {
    if (o->rescoreByPosteriorProbability) return CPECAN_SCORE_BY_POSTERIOR_PROBABILITY;
    if (o->rescoreByPosteriorProbabilityIgnoringGaps) return CPECAN_SCORE_BY_POSTERIOR_PROBABILITY_IGNORING_GAPS;
    if (o->rescoreByIdentity) return CPECAN_SCORE_BY_IDENTITY;
    if (o->rescoreByIdentityIgnoringGaps) return CPECAN_SCORE_BY_IDENTITY_IGNORING_GAPS;
    return -1;
}

/* the realigned alignment of a job, on the forward strands from 0, to its original strands and coordinates and out as cigars
 * (cPecanRealign.c:570-599); consumes rPA */
static void write_alignment(const Job *j, struct PairwiseAlignment *rPA, const Options *o, FILE *out) {
    rebase(&rPA->start1, &rPA->end1, &rPA->strand1, j->shift1, j->flip1);
    rebase(&rPA->start2, &rPA->end2, &rPA->strand2, j->shift2, j->flip2);
    checkPairwiseAlignment(rPA);
    if (o->splitIndelsLongerThanThis != -1) {
        stList *pieces = split_alignment(rPA, o->splitIndelsLongerThanThis);
        for (int64_t i = 0; i < stList_length(pieces); i++) cigarWrite(out, stList_get(pieces, i), 0);
        stList_destruct(pieces);
    } else {
        cigarWrite(out, rPA, 0);
    }
    destructPairwiseAlignment(rPA);
}

/* everything after the device pass for alignment i of the batch (cPecanRealign.c:540-599): the device decoded it (r) */
static void job_finish(Job *j, const CpecanRealignedCigars *r, int64_t i, const Options *o, FILE *out) {
    struct PairwiseAlignment *pA = j->pA;
    if (o->allPosteriorProbsFile != NULL) {
        const int64_t *off = r->rawPairs.offsets;
        write_posterior_probs(o->allPosteriorProbsFile, r->rawPairs.values + 3 * off[i], off[i + 1] - off[i], j);
    }
    if (r->scores != NULL) pA->score = r->scores[i];
    if (o->posteriorProbsFile != NULL) {
        const int64_t *off = r->alignments.offsets;
        write_posterior_probs(o->posteriorProbsFile, r->alignments.values + 3 * off[i], off[i + 1] - off[i], j);
    }
    struct List *ops = constructEmptyList(0, (void (*)(void *)) destructAlignmentOperation);
    for (int64_t k = r->ops.offsets[i]; k < r->ops.offsets[i + 1]; k++) add_op(ops, r->ops.values[2 * k], r->ops.values[2 * k + 1]);
    write_alignment(j, constructPairwiseAlignment(pA->contig1, 0, pA->end1, 1, pA->contig2, 0, pA->end2, 1, pA->score, ops), o, out);
}

/* the same for --rescoreOriginalAlignment: the input columns scored against the posteriors (consumes alignedPairs) */
static void job_finish_rescored(Job *j, stList *alignedPairs, const Options *o, FILE *out) {
    struct PairwiseAlignment *pA = j->pA;
    const int64_t lX = (int64_t) strlen(j->subX), lY = (int64_t) strlen(j->subY);
    if (o->allPosteriorProbsFile != NULL) write_posterior_list(o->allPosteriorProbsFile, alignedPairs, j);
    stList *rescored = score_anchor_pairs(j->anchors, alignedPairs);
    stList_destruct(alignedPairs);
    alignedPairs = rescored;
    if (o->rescoreByPosteriorProbability) pA->score = scoreByPosteriorProbability(lX, lY, alignedPairs);
    else if (o->rescoreByPosteriorProbabilityIgnoringGaps) pA->score = scoreByPosteriorProbabilityIgnoringGaps(alignedPairs);
    else if (o->rescoreByIdentity) pA->score = scoreByIdentity(j->subX, j->subY, lX, lY, alignedPairs);
    else if (o->rescoreByIdentityIgnoringGaps) pA->score = scoreByIdentityIgnoringGaps(j->subX, j->subY, alignedPairs);
    if (o->posteriorProbsFile != NULL) write_posterior_list(o->posteriorProbsFile, alignedPairs, j);
    /* (weight, x, y) -> (x, y), ascending */
    const int64_t nPairs = stList_length(alignedPairs);
    int64_t *xy = xmalloc((size_t) (nPairs > 0 ? nPairs : 1) * 2 * sizeof(int64_t));
    bool ascending = true;
    for (int64_t i = 0; i < nPairs; i++) {
        stIntTuple *t = stList_get(alignedPairs, i);
        xy[2 * i] = stIntTuple_get(t, 1);
        xy[2 * i + 1] = stIntTuple_get(t, 2);
        ascending = ascending && (i == 0 || by_x_then_y(xy + 2 * (i - 1), xy + 2 * i) <= 0);
    }
    stList_destruct(alignedPairs);
    if (!ascending) qsort(xy, (size_t) nPairs, 2 * sizeof(int64_t), by_x_then_y);
    struct PairwiseAlignment *rPA = pairs_to_alignment(pA->contig1, pA->contig2, pA->score, pA->end1, pA->end2, xy, nPairs);
    free(xy);
    write_alignment(j, rPA, o, out);
}

/* the host work on either side of a device pass, over a range of the batch's alignments (cpecan_parallel_for) */
typedef struct {
    Job *jobs;
    stList **pairs;                 /* --rescoreOriginalAlignment: the posteriors of every alignment */
    const CpecanRealignedCigars *r; /* otherwise: the device's realignments */
    char **text;
    const PairwiseAlignmentParameters *p;
    const Options *o;
} HostPass;

static void finish_one(HostPass *h, int64_t i, FILE *out) {
    if (h->pairs != NULL) job_finish_rescored(&h->jobs[i], h->pairs[i], h->o, out);
    else job_finish(&h->jobs[i], h->r, i, h->o, out);
}

static void prepare_range(int64_t first, int64_t last, void *arg) {
    HostPass *h = arg;
    for (int64_t i = first; i < last; i++) job_prepare(&h->jobs[i], h->jobs[i].pA, h->p);
}

static void finish_range(int64_t first, int64_t last, void *arg) {
    HostPass *h = arg;
    for (int64_t i = first; i < last; i++) {
        size_t size = 0;
        FILE *f = open_memstream(&h->text[i], &size);
        if (f == NULL) st_errAbort("cPecanRealign: out of memory");
        finish_one(h, i, f);
        fclose(f);
    }
}

/* $CPECAN_HOST_TIMING: wall-clock time of the program's stages on stderr */
static double g_stageClock;
static bool g_stageTiming;
static double stage_now(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double) ts.tv_sec + 1e-9 * (double) ts.tv_nsec;
}
static void stage(const char *what) {
    if (!g_stageTiming) return;
    const double t = stage_now();
    fprintf(stderr, "[cPecanRealign] %-44s %8.1f ms\n", what, 1e3 * (t - g_stageClock));
    g_stageClock = t;
}

int main(int argc, char *argv[]) {
    g_stageTiming = getenv("CPECAN_HOST_TIMING") != NULL;
    g_stageClock = stage_now();
    PairwiseAlignmentParameters *p = pairwiseAlignmentBandingParameters_construct();
    p->constraintDiagonalTrim = 0; /* the CLI's own defaults (cPecanRealign.c:359-361) */
    p->splitMatrixBiggerThanThis = 10;
    p->diagonalExpansion = 4;
    Options o;
    memset(&o, 0, sizeof(o));
    o.matchGamma = 0.85f;
    o.splitIndelsLongerThanThis = -1;
    const char *expectationsFile = NULL, *hmmFile = NULL;
    int64_t batchBases = 200000000;

    static struct option longOptions[] = { { "logLevel", required_argument, 0, 'a' },
                                           { "help", no_argument, 0, 'h' },
                                           { "gapGamma", required_argument, 0, 'l' },
                                           { "matchGamma", required_argument, 0, 'L' },
                                           { "splitMatrixBiggerThanThis", required_argument, 0, 'o' },
                                           { "diagonalExpansion", required_argument, 0, 'r' },
                                           { "constraintDiagonalTrim", required_argument, 0, 't' },
                                           { "alignAmbiguityCharacters", no_argument, 0, 'w' },
                                           { "rescoreOriginalAlignment", no_argument, 0, 'x' },
                                           { "rescoreByIdentity", no_argument, 0, 'i' },
                                           { "rescoreByPosteriorProb", no_argument, 0, 'j' },
                                           { "rescoreByPosteriorProbIgnoringGaps", no_argument, 0, 'm' },
                                           { "rescoreByIdentityIgnoringGaps", no_argument, 0, 'k' },
                                           { "splitIndelsLongerThanThis", required_argument, 0, 's' },
                                           { "outputPosteriorProbs", required_argument, 0, 'u' },
                                           { "outputAllPosteriorProbs", required_argument, 0, 'z' },
                                           { "outputExpectations", required_argument, 0, 'v' },
                                           { "loadHmm", required_argument, 0, 'y' },
                                           { "batchBases", required_argument, 0, 'b' },
                                           { "gpus", required_argument, 0, 'G' },
                                           { 0, 0, 0, 0 } };
    for (;;) {
        int index = 0;
        const int key = getopt_long(argc, argv, "a:hl:o:r:t:s:wxijkmu:v:y:z:L:b:", longOptions, &index);
        if (key == -1) break;
        switch (key) {
        case 'a': set_log_level(optarg); break;
        case 'h': usage(); return 0;
        case 'l': p->gapGamma = parse_float(optarg, "--gapGamma"); break;
        case 'L': o.matchGamma = parse_float(optarg, "--matchGamma"); break;
        case 'o': {
            const int64_t side = parse_int(optarg, "--splitMatrixBiggerThanThis");
            p->splitMatrixBiggerThanThis = side * side;
            break;
        }
        case 'r':
            p->diagonalExpansion = parse_int(optarg, "--diagonalExpansion");
            if (p->diagonalExpansion % 2 != 0) st_errAbort("cPecanRealign: --diagonalExpansion must be even");
            break;
        case 't': p->constraintDiagonalTrim = parse_int(optarg, "--constraintDiagonalTrim"); break;
        case 'w': p->alignAmbiguityCharacters = 1; break;
        case 'x': o.rescoreOriginalAlignment = 1; break;
        case 'i': o.rescoreByIdentity = 1; break;
        case 'j': o.rescoreByPosteriorProbability = 1; break;
        case 'k': o.rescoreByIdentityIgnoringGaps = 1; break;
        case 'm': o.rescoreByPosteriorProbabilityIgnoringGaps = 1; break;
        case 's': o.splitIndelsLongerThanThis = parse_int(optarg, "--splitIndelsLongerThanThis"); break;
        case 'u': o.posteriorProbsFile = optarg; break;
        case 'v': expectationsFile = optarg; break;
        case 'y': hmmFile = optarg; break;
        case 'z': o.allPosteriorProbsFile = optarg; break;
        case 'b':
            batchBases = parse_int(optarg, "--batchBases");
            if (batchBases == 0) st_errAbort("cPecanRealign: --batchBases must be positive");
            break;
        case 'G': {
            const int64_t gpus = parse_int(optarg, "--gpus");
            if (gpus < 1 || gpus > 16) st_errAbort("cPecanRealign: --gpus takes 1 to 16");
            cpecan_setDevices((int) gpus);
            break;
        }
        default: usage(); return 1;
        }
    }
    log_info("Starting realigning pairwise alignments\n");

    StateMachine *sM;
    if (hmmFile != NULL) {
        log_info("Loading the hmm from file %s\n", hmmFile);
        Hmm *hmm = hmm_loadFromFile(hmmFile);
        sM = hmm_getStateMachine(hmm);
        hmm_destruct(hmm);
    } else {
        sM = stateMachine5_construct(fiveState);
    }
    Hmm *hmmExpectations = expectationsFile != NULL ? hmm_constructEmpty(0.000000000001, sM->type) : NULL; /* the tiny pseudo-count prevents overflow */

    if (optind >= argc) {
        usage();
        return 1;
    }
    read_sequence_files(argc, argv, optind);
    stage("options, model, sequence files");

    /* read a batch of cigars, one device pass, finish and write them in order; repeat */
    Job *jobs = NULL;
    int64_t capJobs = 0;
    bool more = true;
    while (more) {
        int64_t n = 0, bases = 0;
        while (bases < batchBases) {
            struct PairwiseAlignment *pA = cigarRead(stdin);
            if (pA == NULL) {
                more = false;
                break;
            }
            if (n == capJobs) {
                capJobs = capJobs ? 2 * capJobs : 1024;
                jobs = realloc(jobs, (size_t) capJobs * sizeof(Job));
                if (jobs == NULL) st_errAbort("cPecanRealign: out of memory");
            }
            jobs[n].pA = pA; /* prepared below, all alignments of the batch on the host threads together */
            bases += llabs((long long) (pA->end1 - pA->start1)) + llabs((long long) (pA->end2 - pA->start2));
            n++;
        }
        if (n == 0) break;
        stage("cigars of the batch read");
        int64_t *work = xmalloc((size_t) (n + 1) * sizeof(int64_t)); /* prefix sums of the alignments' bases: how the host threads share them */
        work[0] = 0;
        for (int64_t i = 0; i < n; i++) {
            const struct PairwiseAlignment *q = jobs[i].pA;
            work[i + 1] = work[i] + llabs((long long) (q->end1 - q->start1)) + llabs((long long) (q->end2 - q->start2)) + 1;
        }
        {
            HostPass pass = { jobs, NULL, NULL, NULL, p, NULL };
            cpecan_parallel_for(n, work, prepare_range, &pass);
        }
        const char **sX = xmalloc((size_t) n * sizeof(char *)), **sY = xmalloc((size_t) n * sizeof(char *));
        stList **anchors = xmalloc((size_t) n * sizeof(stList *));
        bool *ragged = xmalloc((size_t) n * sizeof(bool));
        for (int64_t i = 0; i < n; i++) {
            sX[i] = jobs[i].subX;
            sY[i] = jobs[i].subY;
            anchors[i] = jobs[i].filtered;
            ragged[i] = 1; /* both ends of a local alignment are ragged (cPecanRealign.c:532, :537) */
        }
        stage("sub-sequences and anchors (host threads)");
        log_info("Device pass over %" PRIi64 " alignments, %" PRIi64 " bases\n", n, bases);
        if (hmmExpectations != NULL) {
            getExpectationsUsingAnchorsBatch(sM, hmmExpectations, n, sX, sY, anchors, p, ragged, ragged);
        } else {
            /* the realignment (cPecanRealign.c:560-569: reweighting, ordered chain, score) and its cigar are built on the device; only
             * --rescoreOriginalAlignment scores the input columns against the posteriors here */
            stList **pairs = NULL;
            CpecanRealignedCigars *r = NULL;
            if (o.rescoreOriginalAlignment) {
                pairs = getAlignedPairsUsingAnchorsBatch(sM, n, sX, sY, anchors, p, ragged, ragged);
                stage("batch call (device pass + lists)");
            } else {
                r = getRealignedCigarsUsingAnchorsBatch(sM, n, sX, sY, anchors, p, ragged, ragged, o.matchGamma, score_kind(&o), o.posteriorProbsFile != NULL,
                                                        o.allPosteriorProbsFile != NULL);
                stage("batch call (device pass, decode, cigars)");
            }
            HostPass pass = { jobs, pairs, r, NULL, p, &o };
            if (o.posteriorProbsFile != NULL || o.allPosteriorProbsFile != NULL) {
                for (int64_t i = 0; i < n; i++) finish_one(&pass, i, stdout); /* each rewrites the files, in input order */
            } else {
                /* everything after the device pass is per alignment: on the host threads, each alignment's cigars into a buffer of
                 * its own, the buffers to the standard output in input order */
                char **text = xmalloc((size_t) n * sizeof(char *));
                pass.text = text;
                cpecan_parallel_for(n, work, finish_range, &pass);
                for (int64_t i = 0; i < n; i++) {
                    fputs(text[i], stdout);
                    free(text[i]);
                }
                free(text);
            }
            free(pairs);
            cpecanRealignedCigars_destruct(r);
            stage("cigars out (host threads)");
        }
        for (int64_t i = 0; i < n; i++) job_release(&jobs[i]);
        free(work);
        free(sX);
        free(sY);
        free(anchors);
        free(ragged);
    }
    free(jobs);

    if (hmmExpectations != NULL) {
        log_info("Writing out expectations to file %s\n", expectationsFile);
        FILE *f = fopen(expectationsFile, "w");
        if (f == NULL) st_errAbort("cPecanRealign: cannot write %s", expectationsFile);
        hmm_write(hmmExpectations, f);
        fclose(f);
        hmm_destruct(hmmExpectations);
    }
    free_sequences();
    stateMachine_destruct(sM);
    pairwiseAlignmentBandingParameters_destruct(p);
    cpecan_shutdown();
    stage("release");
    log_info("Finished realigning pairwise alignments, exiting.\n");
    return 0;
}
