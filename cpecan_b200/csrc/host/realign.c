/*
 * realign.c -- what happens to the posterior-probability pairs after the device pass, for cPecanRealign and for callers
 * that want one alignment rather than a cloud of pairs: anchors from a cigar, AMAP-style gap reweighting, scores, the
 * heaviest ordered chain, the maximal-expected-accuracy alignment and its left shift.  Host-side list work on the compacted
 * output (a few pairs per base); nothing here touches the DP.
 *
 * Reference behaviour followed (citations to the reference tree):
 *   convertPairwiseForwardStrandAlignmentToAnchorPairs   impl/pairwiseAligner.c:979-1003
 *   getIndelProbabilities / reweightAlignedPairs[2]      impl/pairwiseAligner.c:1519-1560
 *   getNumberOfMatchingAlignedPairs / scoreBy*           impl/pairwiseAligner.c:1562-1597
 *   getMaximalExpectedAccuracyPairwiseAlignment          impl/pairwiseAligner.c:1603-1724
 *   leftShiftAlignment / getShiftedMEAAlignment          impl/pairwiseAligner.c:1726-1792
 *   filterPairwiseAlignmentToMakePairsOrdered            impl/multipleAligner.c:945-972 (two-sequence case of the progressive
 *                                                        column aligner, :358-492)
 */
#include <ctype.h>
#include <inttypes.h>
#include <stdbool.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "cpecan/multipleAligner.h"
#include "cpecan/pairwiseAligner.h"
#include "cpecan/pairwiseAlignment.h"
#include "host_internal.h"

static stList *new_tuple_list(void) { return stList_construct3(0, (void (*)(void *)) stIntTuple_destruct); }

/* ---- anchors from a forward-strand cigar: every column of every match run, minus `trim` columns at both ends ---- */

stList *convertPairwiseForwardStrandAlignmentToAnchorPairs(struct PairwiseAlignment *pA, int64_t trim, int64_t diagonalExpansion) {
    if (!pA->strand1 || !pA->strand2) st_errAbort("anchor pairs need a forward-strand alignment (%s / %s)", pA->contig1, pA->contig2);
    /* count first: the tuples of the list then come from one slab (cpecan_tripleList_construct) instead of one allocation per column,
     * which is what a thousand columns per alignment times tens of thousands of alignments spent their time in */
    int64_t n = 0, x = pA->start1, y = pA->start2;
    for (int64_t i = 0; i < pA->operationList->length; i++) {
        const struct AlignmentOperation *op = pA->operationList->list[i];
        if (op->opType == PAIRWISE_MATCH && op->length > 2 * trim) n += op->length - 2 * trim;
        if (op->opType != PAIRWISE_INDEL_Y) x += op->length;
        if (op->opType != PAIRWISE_INDEL_X) y += op->length;
    }
    if (x != pA->end1 || y != pA->end2) st_errAbort("cigar operations of %s / %s do not end at the alignment's end coordinates", pA->contig1, pA->contig2);
    const bool narrow = pA->start1 >= 0 && pA->start2 >= 0 && x <= INT32_MAX && y <= INT32_MAX && diagonalExpansion >= INT32_MIN && diagonalExpansion <= INT32_MAX;
    stList *anchors = narrow ? NULL : new_tuple_list();
    int32_t *flat = narrow ? cpecan_malloc((size_t) (n > 0 ? n : 1) * 3 * sizeof(int32_t)) : NULL;
    int64_t at = 0;
    x = pA->start1;
    y = pA->start2;
    for (int64_t i = 0; i < pA->operationList->length; i++) {
        const struct AlignmentOperation *op = pA->operationList->list[i];
        if (op->opType == PAIRWISE_MATCH) {
            for (int64_t l = trim; l < op->length - trim; l++) {
                if (narrow) {
                    flat[3 * at] = (int32_t) (x + l);
                    flat[3 * at + 1] = (int32_t) (y + l);
                    flat[3 * at + 2] = (int32_t) diagonalExpansion;
                    at++;
                } else {
                    stList_append(anchors, stIntTuple_construct3(x + l, y + l, diagonalExpansion));
                }
            }
        }
        if (op->opType != PAIRWISE_INDEL_Y) x += op->length;
        if (op->opType != PAIRWISE_INDEL_X) y += op->length;
    }
    if (narrow) {
        anchors = cpecan_tripleList_construct(flat, at);
        free(flat);
    }
    return anchors;
}

/* ---- gap reweighting ---- */

int64_t *getIndelProbabilities(stList *alignedPairs, int64_t seqLength, bool xIfTrueElseY) {
    int64_t *gap = cpecan_malloc((size_t) seqLength * sizeof(int64_t));
    for (int64_t i = 0; i < seqLength; i++) gap[i] = PAIR_ALIGNMENT_PROB_1;
    const int64_t n = stList_length(alignedPairs), field = xIfTrueElseY ? 1 : 2;
    for (int64_t i = 0; i < n; i++) {
        stIntTuple *t = stList_get(alignedPairs, i);
        gap[stIntTuple_get(t, field)] -= stIntTuple_get(t, 0);
    }
    for (int64_t i = 0; i < seqLength; i++) {
        if (gap[i] < 0) gap[i] = 0;
    }
    return gap;
}

stList *reweightAlignedPairs(stList *alignedPairs, int64_t *indelProbsX, int64_t *indelProbsY, double gapGamma) {
    stList *out = new_tuple_list();
    const int64_t n = stList_length(alignedPairs);
    for (int64_t i = 0; i < n; i++) {
        stIntTuple *t = stList_get(alignedPairs, i);
        const int64_t x = stIntTuple_get(t, 1), y = stIntTuple_get(t, 2);
        /* integer minus double, truncated towards zero on the way back: the reference's arithmetic (:1547) */
        const int64_t w = (int64_t) ((double) stIntTuple_get(t, 0) - gapGamma * (double) (indelProbsX[x] + indelProbsY[y]));
        stList_append(out, stIntTuple_construct3(w, x, y));
    }
    stList_destruct(alignedPairs);
    return out;
}

stList *reweightAlignedPairs2(stList *alignedPairs, int64_t seqLengthX, int64_t seqLengthY, double gapGamma) {
    if (gapGamma <= 0.0) return alignedPairs;
    int64_t *gX = getIndelProbabilities(alignedPairs, seqLengthX, 1), *gY = getIndelProbabilities(alignedPairs, seqLengthY, 0);
    alignedPairs = reweightAlignedPairs(alignedPairs, gX, gY, gapGamma);
    free(gX);
    free(gY);
    return alignedPairs;
}

/* ---- scores ---- */

int64_t getNumberOfMatchingAlignedPairs(char *subSeqX, char *subSeqY, stList *alignedPairs) {
    int64_t matches = 0;
    const int64_t n = stList_length(alignedPairs);
    for (int64_t i = 0; i < n; i++) {
        stIntTuple *t = stList_get(alignedPairs, i);
        const int cx = toupper((unsigned char) subSeqX[stIntTuple_get(t, 1)]), cy = toupper((unsigned char) subSeqY[stIntTuple_get(t, 2)]);
        matches += cx == cy && cx != 'N';
    }
    return matches;
}

static double total_weight(stList *alignedPairs) {
    double s = 0.0;
    const int64_t n = stList_length(alignedPairs);
    for (int64_t i = 0; i < n; i++) s += (double) stIntTuple_get(stList_get(alignedPairs, i), 0);
    return s;
}

double scoreByIdentity(char *subSeqX, char *subSeqY, int64_t lX, int64_t lY, stList *alignedPairs) {
    const int64_t matches = getNumberOfMatchingAlignedPairs(subSeqX, subSeqY, alignedPairs);
    return 100.0 * ((lX + lY) == 0 ? 0 : (2.0 * matches) / (lX + lY));
}

double scoreByIdentityIgnoringGaps(char *subSeqX, char *subSeqY, stList *alignedPairs) {
    return 100.0 * getNumberOfMatchingAlignedPairs(subSeqX, subSeqY, alignedPairs) / (double) stList_length(alignedPairs);
}

double scoreByPosteriorProbability(int64_t lX, int64_t lY, stList *alignedPairs) {
    return 100.0 * ((lX + lY) == 0 ? 0 : (2.0 * total_weight(alignedPairs)) / ((lX + lY) * PAIR_ALIGNMENT_PROB_1));
}

double scoreByPosteriorProbabilityIgnoringGaps(stList *alignedPairs) {
    return 100.0 * total_weight(alignedPairs) / ((double) stList_length(alignedPairs) * PAIR_ALIGNMENT_PROB_1);
}

/* ---- heaviest ordered chain ----
 * The reference sends the two sequences through its progressive multiple aligner; for two sequences that is a sweep over x
 * keeping a staircase of chain ends (y ascending, score ascending).  Same result with a prefix-maximum tree over y: the best
 * chain ending strictly left of y, ties going to the smaller y and then to the later pair, which is what the staircase keeps
 * (:434-446).  Only pairs with weight/PAIR_ALIGNMENT_PROB_1 >= matchGamma and > 0 take part (:395).  The reference also adds
 * st_random()*1e-5 to every weight (:145) to balance its trees; we do not, so exact ties may resolve differently. */

typedef struct {
    int64_t x, y, w;
    double score; /* weight of the best chain ending here */
    int64_t prev; /* index of the previous pair of that chain, -1 = none */
} ChainPair;

static int chain_by_x_then_y_descending(const void *a, const void *b) {
    const ChainPair *p = a, *q = b;
    if (p->x != q->x) return p->x < q->x ? -1 : 1;
    return p->y > q->y ? -1 : (p->y < q->y ? 1 : 0);
}

/* is chain end a better than chain end b?  (-1 = no chain) */
static bool chain_better(const ChainPair *c, int64_t a, int64_t b) {
    if (b < 0) return a >= 0;
    if (a < 0) return false;
    if (c[a].score != c[b].score) return c[a].score > c[b].score;
    if (c[a].y != c[b].y) return c[a].y < c[b].y;
    return a > b;
}

stList *filterPairwiseAlignmentToMakePairsOrdered(stList *alignedPairs, const char *seqX, const char *seqY, float matchGamma) {
    (void) seqX;
    const int64_t n = stList_length(alignedPairs), lY = (int64_t) strlen(seqY);
    ChainPair *c = cpecan_malloc((size_t) (n + 1) * sizeof(ChainPair));
    int64_t m = 0;
    for (int64_t i = 0; i < n; i++) {
        stIntTuple *t = stList_get(alignedPairs, i);
        const double w = (double) stIntTuple_get(t, 0) / PAIR_ALIGNMENT_PROB_1;
        if (w >= matchGamma && w > 0.0) {
            c[m].w = stIntTuple_get(t, 0);
            c[m].x = stIntTuple_get(t, 1);
            c[m].y = stIntTuple_get(t, 2);
            if (c[m].y < 0 || c[m].y >= lY) st_errAbort("aligned pair (%" PRIi64 ", %" PRIi64 ") lies outside sequence Y", c[m].x, c[m].y);
            m++;
        }
    }
    qsort(c, (size_t) m, sizeof(ChainPair), chain_by_x_then_y_descending);
    /* tree[k] = best chain end among the y positions the Fenwick node k covers */
    int64_t *tree = cpecan_malloc((size_t) (lY + 1) * sizeof(int64_t));
    for (int64_t k = 0; k <= lY; k++) tree[k] = -1;
    int64_t best = -1;
    for (int64_t i = 0; i < m;) {
        int64_t j = i;
        while (j < m && c[j].x == c[i].x) j++;
        /* pairs of one x see only chains that end at smaller x: look all of them up before adding any */
        for (int64_t k = i; k < j; k++) {
            int64_t p = -1;
            for (int64_t f = c[k].y; f > 0; f -= f & -f) { /* prefix [0, y) */
                if (chain_better(c, tree[f], p)) p = tree[f];
            }
            c[k].prev = p;
            c[k].score = (p >= 0 ? c[p].score : 0.0) + (double) c[k].w / PAIR_ALIGNMENT_PROB_1;
        }
        for (int64_t k = i; k < j; k++) { /* y descending, as the reference inserts them */
            for (int64_t f = c[k].y + 1; f <= lY; f += f & -f) {
                if (chain_better(c, k, tree[f])) tree[f] = k;
            }
            if (chain_better(c, k, best)) best = k;
        }
        i = j;
    }
    /* the chain, first pair first; its tuples from one slab when the coordinates allow (they do for anything the device aligned) */
    int64_t len = 0;
    bool narrow = true;
    for (int64_t k = best; k >= 0; k = c[k].prev) {
        len++;
        narrow = narrow && c[k].x >= INT32_MIN && c[k].x <= INT32_MAX && c[k].y <= INT32_MAX && c[k].w >= INT32_MIN && c[k].w <= INT32_MAX;
    }
    stList *out;
    if (narrow) {
        int32_t *flat = cpecan_malloc((size_t) (len > 0 ? len : 1) * 3 * sizeof(int32_t));
        int64_t at = len;
        for (int64_t k = best; k >= 0; k = c[k].prev) {
            at--;
            flat[3 * at] = (int32_t) c[k].w;
            flat[3 * at + 1] = (int32_t) c[k].x;
            flat[3 * at + 2] = (int32_t) c[k].y;
        }
        out = cpecan_tripleList_construct(flat, len);
        free(flat);
    } else {
        out = new_tuple_list();
        for (int64_t k = best; k >= 0; k = c[k].prev) stList_append(out, stIntTuple_construct3(c[k].w, c[k].x, c[k].y));
        stList_reverse(out);
    }
    free(tree);
    free(c);
    stList_destruct(alignedPairs);
    return out;
}

/* ---- maximal expected accuracy ---- */

/* cum[i] = sum of the gap weights of positions 0..i */
static int64_t *cumulative_gap_weights(stList *gapPairs, int64_t seqLength, int field) {
    int64_t *cum = cpecan_malloc((size_t) (seqLength > 0 ? seqLength : 1) * sizeof(int64_t));
    memset(cum, 0, (size_t) (seqLength > 0 ? seqLength : 1) * sizeof(int64_t));
    const int64_t n = stList_length(gapPairs);
    for (int64_t i = 0; i < n; i++) {
        stIntTuple *t = stList_get(gapPairs, i);
        const int64_t pos = stIntTuple_get(t, field);
        if (pos < 0 || pos >= seqLength) st_errAbort("gap pair position %" PRIi64 " lies outside a sequence of length %" PRIi64, pos, seqLength);
        cum[pos] += stIntTuple_get(t, 0);
    }
    for (int64_t i = 1; i < seqLength; i++) cum[i] += cum[i - 1];
    return cum;
}

static int64_t gap_weight(const int64_t *cum, int64_t start, int64_t length) {
    return length == 0 ? 0 : cum[start + length - 1] - (start > 0 ? cum[start - 1] : 0);
}

/* The walk-back from pair (x, y) acts only on entries with x2 < x and y2 < y; every other entry is passed over without effect.  So a range
 * of list positions whose least x is not below x, or whose least y is not below y, holds no predecessor and is skipped whole: score, from,
 * the cutoff and isHigh come out as the entry-by-entry scan leaves them, in any list order.  In the reference's order a region's
 * traceback blocks come last to first, so the walk from a pair of block k would otherwise read every triple of the blocks after k (later
 * diagonals, none of them a predecessor) -- quadratic in the list length.  The least x and y are kept for every aligned range of
 * MEA_CHUNK entries and of MEA_CHUNK^2 entries (decode_kernels.cuh keeps the same two levels). */
#define MEA_CHUNK_SHIFT 5
#define MEA_CHUNK ((int64_t) 1 << MEA_CHUNK_SHIFT)
#define MEA_BLOCK_SHIFT (2 * MEA_CHUNK_SHIFT)
#define MEA_BLOCK ((int64_t) 1 << MEA_BLOCK_SHIFT)

/* least[2 * r], least[2 * r + 1] = the least x and y of the entries r << shift ... ((r + 1) << shift) - 1 */
static int64_t *least_xy(const int64_t *x, const int64_t *y, int64_t n, int shift) {
    const int64_t ranges = (n + ((int64_t) 1 << shift) - 1) >> shift;
    int64_t *least = cpecan_malloc((size_t) (2 * ranges + 2) * sizeof(int64_t));
    for (int64_t r = 0; r < ranges; r++) least[2 * r] = least[2 * r + 1] = INT64_MAX;
    for (int64_t j = 0; j < n; j++) {
        int64_t *l = least + 2 * (j >> shift);
        if (x[j] < l[0]) l[0] = x[j];
        if (y[j] < l[1]) l[1] = y[j];
    }
    return least;
}

stList *getMaximalExpectedAccuracyPairwiseAlignment(stList *alignedPairs, stList *gapXPairs, stList *gapYPairs, int64_t seqXLength,
                                                    int64_t seqYLength, double *alignmentScore, PairwiseAlignmentParameters *p) {
    const int64_t n = stList_length(alignedPairs);
    double *scores = cpecan_malloc((size_t) (n + 1) * sizeof(double));
    int64_t *back = cpecan_malloc((size_t) (n + 1) * sizeof(int64_t));
    bool *isHigh = cpecan_malloc((size_t) (n + 1) * sizeof(bool));
    memset(isHigh, 0, (size_t) (n + 1) * sizeof(bool));
    int64_t *cumY = cumulative_gap_weights(gapYPairs, seqYLength, 2), *cumX = cumulative_gap_weights(gapXPairs, seqXLength, 1);
    int64_t *tw = cpecan_malloc((size_t) (n + 1) * sizeof(int64_t)), *tx = cpecan_malloc((size_t) (n + 1) * sizeof(int64_t)),
            *ty = cpecan_malloc((size_t) (n + 1) * sizeof(int64_t));
    for (int64_t i = 0; i < n; i++) {
        stIntTuple *t = stList_get(alignedPairs, i);
        tw[i] = stIntTuple_get(t, 0);
        tx[i] = stIntTuple_get(t, 1);
        ty[i] = stIntTuple_get(t, 2);
    }
    int64_t *chunk = least_xy(tx, ty, n, MEA_CHUNK_SHIFT), *block = least_xy(tx, ty, n, MEA_BLOCK_SHIFT);
    const float gamma = p->gapGamma;
    double maxScore = 0;
    /* pairs in list order (the engine's order: increasing x + y within a region); a virtual pair at (lX, lY) closes the alignment */
    for (int64_t i = 0; i <= n; i++) {
        int64_t w = 0, x = seqXLength, y = seqYLength;
        if (i < n) {
            w = tw[i];
            x = tx[i];
            y = ty[i];
        }
        double score = w + (gap_weight(cumX, 0, x) + gap_weight(cumY, 0, y)) * gamma;
        int64_t from = -1;
        for (int64_t j = i - 1; j >= 0; j--) {
            /* at the last entry of an aligned range: skip the whole range if it holds no predecessor (a range that i - 1 ends early is scanned) */
            if ((j & (MEA_BLOCK - 1)) == MEA_BLOCK - 1 && !(block[2 * (j >> MEA_BLOCK_SHIFT)] < x && block[2 * (j >> MEA_BLOCK_SHIFT) + 1] < y)) {
                j -= MEA_BLOCK - 1;
                continue;
            }
            if ((j & (MEA_CHUNK - 1)) == MEA_CHUNK - 1 && !(chunk[2 * (j >> MEA_CHUNK_SHIFT)] < x && chunk[2 * (j >> MEA_CHUNK_SHIFT) + 1] < y)) {
                j -= MEA_CHUNK - 1;
                continue;
            }
            const int64_t x2 = tx[j], y2 = ty[j];
            if (x2 < x && y2 < y) {
                /* the candidate is held in an int64 in the reference (:1668), i.e. truncated before the comparison */
                const int64_t s = (int64_t) (w + scores[j] + (gap_weight(cumX, x2 + 1, x - x2 - 1) + gap_weight(cumY, y2 + 1, y - y2 - 1)) * gamma);
                if (s > score) {
                    score = (double) s;
                    from = j;
                }
                if (isHigh[j]) break; /* nothing further back can beat a running maximum */
            }
        }
        back[i] = from;
        scores[i] = score;
        const double s = score + ((x < seqXLength ? gap_weight(cumX, x + 1, seqXLength - x - 1) : 0) +
                                  (y < seqYLength ? gap_weight(cumY, y + 1, seqYLength - y - 1) : 0)) * gamma;
        if (s >= maxScore) {
            maxScore = s;
            isHigh[i] = 1;
        }
    }
    stList *out = new_tuple_list();
    for (int64_t i = back[n]; i >= 0; i = back[i]) {
        stIntTuple *t = stList_get(alignedPairs, i);
        stList_append(out, stIntTuple_construct3(stIntTuple_get(t, 0), stIntTuple_get(t, 1), stIntTuple_get(t, 2)));
    }
    stList_reverse(out);
    free(scores);
    free(back);
    free(isHigh);
    free(tw);
    free(tx);
    free(ty);
    free(chunk);
    free(block);
    free(cumX);
    free(cumY);
    *alignmentScore = maxScore;
    return out;
}

/* ---- left shift: slide matches left through every gap as long as the bases to the left of the gap agree ---- */

stList *leftShiftAlignment(stList *alignedPairs, char *seqX, char *seqY) {
    stList *out = new_tuple_list();
    int64_t x = (int64_t) strlen(seqX), y = (int64_t) strlen(seqY);
    for (int64_t i = stList_length(alignedPairs) - 1; i >= 0; i--) {
        stIntTuple *t = stList_get(alignedPairs, i);
        const int64_t w = stIntTuple_get(t, 0), x2 = stIntTuple_get(t, 1), y2 = stIntTuple_get(t, 2);
        while ((x - x2 > 1 || y - y2 > 1) && toupper((unsigned char) seqX[x - 1]) == toupper((unsigned char) seqY[y - 1])) {
            stList_append(out, stIntTuple_construct3(w, x - 1, y - 1)); /* the shifted match borrows this pair's weight */
            x--;
            y--;
            if (x2 == x || y2 == y) break; /* ran over the pair itself */
        }
        if (x2 < x && y2 < y) {
            stList_append(out, stIntTuple_construct3(w, x2, y2));
            x = x2;
            y = y2;
        }
    }
    while (x > 0 && y > 0 && toupper((unsigned char) seqX[x - 1]) == toupper((unsigned char) seqY[y - 1])) {
        const int64_t w = stList_length(alignedPairs) > 0 ? stIntTuple_get(stList_get(alignedPairs, 0), 0) : 1;
        stList_append(out, stIntTuple_construct3(w, x - 1, y - 1));
        x--;
        y--;
    }
    stList_reverse(out);
    return out;
}

stList *getShiftedMEAAlignment(char *seqX, char *seqY, stList *anchorAlignment, PairwiseAlignmentParameters *p, StateMachine *sM,
                               bool alignmentHasRaggedLeftEnd, bool alignmentHasRaggedRightEnd, double *alignmentScore) {
    stList *alignedPairs, *gapXPairs, *gapYPairs;
    getAlignedPairsWithIndelsUsingAnchors(sM, seqX, seqY, anchorAlignment, p, &alignedPairs, &gapXPairs, &gapYPairs, alignmentHasRaggedLeftEnd,
                                          alignmentHasRaggedRightEnd);
    stList *mea = getMaximalExpectedAccuracyPairwiseAlignment(alignedPairs, gapXPairs, gapYPairs, (int64_t) strlen(seqX), (int64_t) strlen(seqY),
                                                              alignmentScore, p);
    stList *shifted = leftShiftAlignment(mea, seqX, seqY);
    stList_destruct(gapXPairs);
    stList_destruct(gapYPairs);
    stList_destruct(alignedPairs);
    stList_destruct(mea);
    return shifted;
}
