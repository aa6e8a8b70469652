/*
 * anchor_kernels.cuh -- the anchors of getBlastPairsForPairwiseAlignmentParameters (host/anchors.c) on the device, batched over every
 * problem of a chunk (cpb_batch_create_anchored in engine.cu).  A problem is one rectangle of one pair: the whole matrix (level 1) or
 * a gap between two level-1 anchors that is still bigger than anchorMatrixBiggerThanThis (level 2).  The kernels read the RAW bytes
 * of the sequences: the soft mask (lower case) is part of the input.
 *
 *   k_anchor_index      a thread per Y start position: every whole k-mer into the problem's open-addressing table (atomicCAS on the
 *                       key, an atomic count, the largest start): whether a k-mer is unique does not depend on the insertion order
 *   k_anchor_hits       a thread per X start position: the Y position of its k-mer if that k-mer occurs exactly once in Y, else -1
 *   k_anchor_seed_flags a hit starts a seed unless the previous X position hit the previous Y position (anchors.c:141-154)
 *   (scan of the flags)
 *   k_anchor_seeds      a thread per seed start: the seed's length is k plus the hits that extend it
 *   k_anchor_chain      a thread per problem: chain_seeds of anchors.c as written (stable release order of x ends, a Fenwick tree of
 *                       prefix maxima keyed by y end, strict comparisons, the first strict maximum), then the runs count pass
 *   (scan of the counts)
 *   k_anchor_runs       a thread per problem: the runs' triples (x, y, expansion), shifted by the problem's corner
 *   k_anchor_gap_flags / k_anchor_gap_list    level 2: the gaps of every pair's level-1 list that are problems themselves
 *   k_anchor_slot_sizes / k_anchor_merge_*    per pair: gap anchors, then the level-1 anchor, ... then the last gap's anchors
 */
#pragma once
#include <cstdint>

namespace cpb {

struct AnchorProblem {
    int64_t x, y;       /* the problem's first byte in the raw X / Y arrays */
    int64_t xPos, yPos; /* first entry of its per-X-position and per-Y-position arrays in the chunk; yPos counts lY + 2 per problem */
    int64_t tab;        /* first entry of its k-mer table in the chunk */
    int32_t lX, lY, k, mask;
    int32_t dx, dy;     /* added to the output coordinates: the problem's corner in its pair */
    int32_t capMask;    /* table entries - 1 (a power of two >= 2 lY) */
    int32_t pad_;
};

struct KmerEntry {        /* all bytes 0xFF = empty */
    unsigned long long key;
    int32_t count;        /* occurrences - 1 */
    int32_t pos;          /* largest start of the k-mer in Y (the only one where count == 0) */
};

struct AnchorGap {        /* a level-2 problem: rectangle [x, x + lX) x [y, y + lY) of pair `pair`, found at gap slot `slot` */
    int64_t slot;
    int32_t pair, x, y, lX, lY, mask;
};

constexpr unsigned long long kKmerEmpty = ~0ull;

__device__ __forceinline__ int anchor_code(uint8_t ch, int mask) {
    switch (ch) {
    case 'A': return 0;
    case 'C': return 1;
    case 'G': return 2;
    case 'T': return 3;
    case 'a': return mask ? -1 : 0;
    case 'c': return mask ? -1 : 1;
    case 'g': return mask ? -1 : 2;
    case 't': return mask ? -1 : 3;
    default: return -1;
    }
}

__device__ __forceinline__ unsigned long long anchor_mix(unsigned long long k) {
    k ^= k >> 33;
    k *= 0xFF51AFD7ED558CCDull;
    k ^= k >> 33;
    return k;
}

/* the k-mer starting at s[0], or kKmerEmpty if one of its bases is not a valid code */
__device__ __forceinline__ unsigned long long anchor_word(const uint8_t *s, int k, int mask) {
    unsigned long long w = 0;
    for (int j = 0; j < k; j++) {
        const int c = anchor_code(s[j], mask);
        if (c < 0) return kKmerEmpty;
        w = (w << 2) | (unsigned long long) c;
    }
    return w;
}

/* the problem whose range [start(p), start(p + 1)) holds position t: bisection over the chunk's problems */
template <class Start> __device__ __forceinline__ int anchor_problem_of(int64_t t, int nProblems, Start start) {
    int lo = 0, hi = nProblems - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (start(mid) <= t) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

__global__ void k_anchor_index(const AnchorProblem *pr, int nProblems, int64_t totalY, const uint8_t *symY, KmerEntry *table) {
    const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= totalY) return;
    const int p = anchor_problem_of(t, nProblems, [&](int q) { return pr[q].yPos; });
    const AnchorProblem P = pr[p];
    const int64_t y = t - P.yPos;
    if (y + P.k > P.lY) return;
    const unsigned long long w = anchor_word(symY + P.y + y, P.k, P.mask);
    if (w == kKmerEmpty) return;
    KmerEntry *tab = table + P.tab;
    unsigned long long h = anchor_mix(w) & (unsigned long long) P.capMask;
    for (;;) {
        const unsigned long long prev = atomicCAS(&tab[h].key, kKmerEmpty, w);
        if (prev == kKmerEmpty || prev == w) {
            atomicAdd(&tab[h].count, 1);
            atomicMax(&tab[h].pos, (int32_t) y);
            return;
        }
        h = (h + 1) & (unsigned long long) P.capMask;
    }
}

__global__ void k_anchor_hits(const AnchorProblem *pr, int nProblems, int64_t totalX, const uint8_t *symX, const KmerEntry *table, int32_t *hitY) {
    const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= totalX) return;
    const int p = anchor_problem_of(t, nProblems, [&](int q) { return pr[q].xPos; });
    const AnchorProblem P = pr[p];
    const int64_t x = t - P.xPos;
    int32_t hit = -1;
    if (x + P.k <= P.lX && P.lY >= P.k) {
        const unsigned long long w = anchor_word(symX + P.x + x, P.k, P.mask);
        if (w != kKmerEmpty) {
            const KmerEntry *tab = table + P.tab;
            unsigned long long h = anchor_mix(w) & (unsigned long long) P.capMask;
            while (tab[h].key != kKmerEmpty && tab[h].key != w) h = (h + 1) & (unsigned long long) P.capMask;
            if (tab[h].key == w && tab[h].count == 0) hit = tab[h].pos;
        }
    }
    hitY[t] = hit;
}

__global__ void k_anchor_seed_flags(const AnchorProblem *pr, int nProblems, int64_t totalX, const int32_t *hitY, int32_t *flags) {
    const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= totalX) return;
    const int p = anchor_problem_of(t, nProblems, [&](int q) { return pr[q].xPos; });
    const int32_t h = hitY[t];
    flags[t] = h >= 0 && !(t > pr[p].xPos && hitY[t - 1] >= 0 && hitY[t - 1] == h - 1);
}

__global__ void k_anchor_seeds(const AnchorProblem *pr, int nProblems, int64_t totalX, const int32_t *hitY, const int32_t *flags,
                               const int64_t *seedOff, int3 *seeds) {
    const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= totalX || !flags[t]) return;
    const int p = anchor_problem_of(t, nProblems, [&](int q) { return pr[q].xPos; });
    const AnchorProblem P = pr[p];
    const int32_t x = (int32_t) (t - P.xPos), y = hitY[t];
    int32_t j = 1; /* hits (x + j, y + j) extend the seed */
    while (x + j + P.k <= P.lX && hitY[t + j] == y + j) j++;
    seeds[seedOff[t]] = make_int3(x, y, P.k + j - 1);
}

__device__ __forceinline__ bool anchor_same_base(uint8_t p, uint8_t q) {
    const int u = anchor_code(p, 0);
    return u >= 0 && u == anchor_code(q, 0);
}

/* the runs of a chain (anchors.c:272-291): counts the triples, or writes them to out */
template <bool WRITE>
__device__ int64_t anchor_runs(const AnchorProblem &P, const uint8_t *sX, const uint8_t *sY, const int3 *seeds, const int32_t *chain, int32_t m,
                               int64_t trim, int32_t expansion, int32_t *out) {
    int64_t n = 0;
    int32_t i = 0;
    while (i < m) {
        const int3 a = seeds[chain[i]];
        const int64_t x0 = a.x, y0 = a.y, d = x0 - y0;
        int64_t x1 = x0 + a.z;
        int32_t j = i + 1;
        while (j < m) {
            const int3 c = seeds[chain[j]];
            if ((int64_t) c.x - c.y != d) break;
            const int64_t gap = c.x - x1;
            int64_t same = 0;
            for (int64_t t = 0; t < gap; t++) same += anchor_same_base(sX[x1 + t], sY[x1 + t - d]);
            if (10 * same < 6 * gap) break;
            x1 = (int64_t) c.x + c.z;
            j++;
        }
        if (j - i > 1 || x1 - x0 >= 2 * P.k) {
            for (int64_t l = trim; l < x1 - x0 - trim; l++) {
                if (WRITE) {
                    out[3 * n] = (int32_t) (x0 + l + P.dx);
                    out[3 * n + 1] = (int32_t) (y0 + l + P.dy);
                    out[3 * n + 2] = expansion;
                }
                n++;
            }
        }
        i = j;
    }
    return n;
}

/* chain_seeds of anchors.c (:164-222), one thread per problem; score, prev and order are per-seed scratch, fenScore / fenWho per-Y
 * scratch (zeroed; fenWho holds the seed index + 1).  order ends up holding the chain.  Then the runs count pass. */
__global__ void k_anchor_chain(const AnchorProblem *pr, int nProblems, const uint8_t *symX, const uint8_t *symY, const int64_t *seedOff,
                               const int3 *seeds, int32_t *score, int32_t *prev, int32_t *order, int32_t *fenScore, int32_t *fenWho, int64_t trim,
                               int32_t *chainLen, int32_t *counts) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nProblems) return;
    const AnchorProblem P = pr[p];
    const int64_t s0 = seedOff[P.xPos];
    const int32_t n = (int32_t) (seedOff[P.xPos + P.lX] - s0);
    const int3 *sd = seeds + s0;
    int32_t *sc = score + s0, *pv = prev + s0, *byEnd = order + s0;
    int32_t *tS = fenScore + P.yPos, *tW = fenWho + P.yPos;
    const int64_t lY = P.lY;
    for (int32_t i = 0; i < n; i++) { /* stable insertion sort by x end */
        const int64_t e = (int64_t) sd[i].x + sd[i].z;
        int32_t j = i - 1;
        while (j >= 0 && (int64_t) sd[byEnd[j]].x + sd[byEnd[j]].z > e) {
            byEnd[j + 1] = byEnd[j];
            j--;
        }
        byEnd[j + 1] = i;
    }
    int32_t released = 0, bestEnd = -1, bestScore = 0;
    for (int32_t i = 0; i < n; i++) {
        while (released < n && (int64_t) sd[byEnd[released]].x + sd[byEnd[released]].z <= sd[i].x) {
            const int32_t v = byEnd[released++];
            for (int64_t t = (int64_t) sd[v].y + sd[v].z; t <= lY + 1; t += t & -t) {
                if (sc[v] > tS[t]) {
                    tS[t] = sc[v];
                    tW[t] = v + 1;
                }
            }
        }
        int32_t s = 0, who = -1;
        for (int64_t t = sd[i].y; t > 0; t -= t & -t) {
            if (tS[t] > s) {
                s = tS[t];
                who = tW[t] - 1;
            }
        }
        sc[i] = s + sd[i].z;
        pv[i] = who;
        if (sc[i] > bestScore) {
            bestScore = sc[i];
            bestEnd = i;
        }
    }
    int32_t m = 0;
    for (int32_t v = bestEnd; v >= 0; v = pv[v]) m++;
    int32_t at = m;
    for (int32_t v = bestEnd; v >= 0; v = pv[v]) byEnd[--at] = v; /* the release order is no longer needed */
    chainLen[p] = m;
    counts[p] = (int32_t) anchor_runs<false>(P, symX + P.x, symY + P.y, sd, byEnd, m, trim, 0, nullptr);
}

__global__ void k_anchor_runs(const AnchorProblem *pr, int nProblems, const uint8_t *symX, const uint8_t *symY, const int64_t *seedOff,
                              const int3 *seeds, const int32_t *chain, const int32_t *chainLen, int64_t trim, int32_t expansion,
                              const int64_t *outOff, int32_t *out) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nProblems) return;
    const AnchorProblem P = pr[p];
    const int64_t s0 = seedOff[P.xPos];
    anchor_runs<true>(P, symX + P.x, symY + P.y, seeds + s0, chain + s0, chainLen[p], trim, expansion, out + 3 * outOff[p]);
}

/* ---- level 2 (anchors.c:348-381).  Level-1 problem p (pair pairOf[p], lengths lX[p], lY[p]) has off[p + 1] - off[p] anchors and
 * one gap more: gap g lies before anchor g, the last one after the last anchor.  Gap slot off[p] + p + g numbers them all. ---- */
__device__ __forceinline__ void anchor_gap_of(int64_t s, int nProblems, const int64_t *off, const int32_t *tri, const int32_t *lX,
                                              const int32_t *lY, int *pOut, int64_t *gOut, int64_t *rect) {
    const int p = anchor_problem_of(s, nProblems, [&](int q) { return off[q] + q; });
    const int64_t g = s - off[p] - p, n1 = off[p + 1] - off[p];
    const int32_t *a = tri + 3 * off[p];
    rect[0] = g > 0 ? (int64_t) a[3 * (g - 1)] + 1 : 0;
    rect[1] = g > 0 ? (int64_t) a[3 * (g - 1) + 1] + 1 : 0;
    rect[2] = g < n1 ? (int64_t) a[3 * g] : lX[p];
    rect[3] = g < n1 ? (int64_t) a[3 * g + 1] : lY[p];
    *pOut = p;
    *gOut = g;
}

__global__ void k_anchor_gap_flags(int nProblems, const int64_t *off, const int32_t *tri, const int32_t *lX, const int32_t *lY, int64_t nSlots,
                                   long long anchorBiggerThan, int32_t *flags) {
    const int64_t s = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nSlots) return;
    int p;
    int64_t g, r[4];
    anchor_gap_of(s, nProblems, off, tri, lX, lY, &p, &g, r);
    const int64_t w = r[2] - r[0], h = r[3] - r[1];
    flags[s] = w > 0 && h > 0 && w * h > anchorBiggerThan;
}

__global__ void k_anchor_gap_list(int nProblems, const int64_t *off, const int32_t *tri, const int32_t *lX, const int32_t *lY, const int32_t *pairOf,
                                  int64_t nSlots, long long maskBiggerThan, const int32_t *flags, const int64_t *gapIdx, AnchorGap *gaps) {
    const int64_t s = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nSlots || !flags[s]) return;
    int p;
    int64_t g, r[4];
    anchor_gap_of(s, nProblems, off, tri, lX, lY, &p, &g, r);
    AnchorGap G;
    G.slot = s;
    G.pair = pairOf[p];
    G.x = (int32_t) r[0];
    G.y = (int32_t) r[1];
    G.lX = (int32_t) (r[2] - r[0]);
    G.lY = (int32_t) (r[3] - r[1]);
    G.mask = (r[2] - r[0]) * (r[3] - r[1]) > maskBiggerThan;
    gaps[gapIdx[s]] = G;
}

/* triples each gap slot contributes to its pair's list: the gap's own anchors and the level-1 anchor after it (none after the last) */
__global__ void k_anchor_slot_sizes(int nProblems, const int64_t *off, int64_t nSlots, const int32_t *flags, const int64_t *gapIdx, const int64_t *gapOff,
                                    int32_t *sizes) {
    const int64_t s = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nSlots) return;
    const int p = anchor_problem_of(s, nProblems, [&](int q) { return off[q] + q; });
    const int64_t g = s - off[p] - p;
    int64_t n = g < off[p + 1] - off[p] ? 1 : 0;
    if (flags != nullptr && flags[s]) n += gapOff[gapIdx[s] + 1] - gapOff[gapIdx[s]];
    sizes[s] = (int32_t) n;
}

__global__ void k_anchor_merge_level1(int nProblems, const int64_t *off, const int32_t *tri, int64_t nSlots, const int32_t *flags, const int64_t *gapIdx,
                                      const int64_t *gapOff, const int64_t *slotPos, int32_t *out) {
    const int64_t s = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nSlots) return;
    const int p = anchor_problem_of(s, nProblems, [&](int q) { return off[q] + q; });
    const int64_t g = s - off[p] - p;
    if (g >= off[p + 1] - off[p]) return;
    int64_t at = slotPos[s];
    if (flags != nullptr && flags[s]) at += gapOff[gapIdx[s] + 1] - gapOff[gapIdx[s]];
    const int32_t *a = tri + 3 * (off[p] + g);
    out[3 * at] = a[0];
    out[3 * at + 1] = a[1];
    out[3 * at + 2] = a[2];
}

__global__ void k_anchor_merge_level2(int nGaps, const AnchorGap *gaps, const int64_t *gapOff, const int32_t *tri, const int64_t *slotPos, int32_t *out) {
    const int64_t j = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= gapOff[nGaps]) return;
    const int q = anchor_problem_of(j, nGaps, [&](int r) { return gapOff[r]; });
    const int64_t at = slotPos[gaps[q].slot] + (j - gapOff[q]);
    out[3 * at] = tri[3 * j];
    out[3 * at + 1] = tri[3 * j + 1];
    out[3 * at + 2] = tri[3 * j + 2];
}

/* anchors per pair: the span of its level-1 problem's gap slots (pairs without a problem have none) */
__global__ void k_anchor_pair_counts(int nPairs, const int32_t *problemOf, const int64_t *off, const int64_t *slotPos, int32_t *counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nPairs) return;
    const int p = problemOf[i];
    counts[i] = p < 0 ? 0 : (int32_t) (slotPos[off[p + 1] + p + 1] - slotPos[off[p] + p]);
}

} // namespace cpb
