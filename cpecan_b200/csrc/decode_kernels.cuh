/*
 * decode_kernels.cuh -- posteriors to one alignment per pair on the device: the heaviest ordered chain, the maximal-expected-accuracy
 * alignment with its left shift, and the four scores of an alignment.  Each kernel restates a host function of host/realign.c and gives
 * the same triples in the same order, with the same double bits:
 *
 *   k_chain_sort / k_chain_sweep / k_chain_write   filterPairwiseAlignmentToMakePairsOrdered   realign.c:150-247
 *   k_ref_order (k_ref_emit)                       cpb_batch_fetch_pairs_reference_order (the order libcpecan.so hands lists over in)
 *   k_mea_gaps / k_mea_summaries / k_mea           getMaximalExpectedAccuracyPairwiseAlignment realign.c:249-371
 *   k_decode_emit<SHIFT>                           its traceback, and leftShiftAlignment        realign.c:353-358, :375-401
 *   k_decode_scores                                scoreByIdentity ... IgnoringGaps             realign.c:113-148
 *   k_reanchor_count / k_reanchor_write            the anchors job_prepare builds from the cigar of an alignment (realignJobs.h:149-173,
 *                                                  realign.c:32-72, cPecanRealign.c:98-123)
 *   k_cigar_count / k_cigar_write                  the cigar operations cPecanRealign writes for an alignment (pairs_to_alignment,
 *                                                  cPecanRealign.c:98-123)
 *   k_cigar_cols_count / k_cigar_cols_write<true>  the anchors job_prepare builds from an input cigar (realignJobs.h:149-173, realign.c:32-72)
 *   k_cigar_cols_write<false> / k_cigar_weigh      an input cigar's columns weighed against list 0 (score_anchor_pairs, cPecanRealign.c:78-104)
 *
 * Pairs are processed in chunks whose work arrays fit the context's scratch budget (engine.cu); DecodePair says where a pair's inputs
 * and work arrays are.  Alignments are int32 (pInt, x, y) triples, 0-based, like the result lists.
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "cpecan_b200.h"

namespace cpb {

struct DecodePair {
    int64_t list0, gap1, gap2; /* first triple of the pair in lists 0, 1, 2 (device order) */
    int64_t seqX, seqY;        /* first byte of the pair in the kept (upper-cased) sequence bytes */
    int64_t work;              /* byte offset of the pair's work arrays in the chunk's scratch */
    int64_t region0, region1;  /* the pair's regions of the last run, [region0, region1) (MEA) */
    int32_t n0, n1, n2;
    int32_t lX, lY;
    int32_t pad_;
};

__host__ __device__ __forceinline__ int64_t dec_round(int64_t bytes) { return (bytes + 15) & ~(int64_t) 15; }

/* ---- heaviest ordered chain ----
 * Work arrays of a pair with m triples in list 0: per x the number of taking-part triples (then the end of its bucket), the triples
 * sorted by x ascending and y descending, their chain scores and predecessors, and a Fenwick tree over y whose nodes hold the best
 * chain end (score, y, sorted index) of the positions they cover. */
struct ChainNode {
    double score;
    int32_t y, idx; /* idx -1: no chain */
};

__host__ __device__ __forceinline__ int64_t chain_work_bytes(int64_t m, int64_t lX, int64_t lY) {
    return dec_round(4 * (lX + 1)) + dec_round(12 * m) + dec_round(8 * m) + dec_round(4 * m) + dec_round(16 * (lY + 1)) + 16;
}

struct ChainWork {
    int32_t *count;
    int3 *ent; /* (x, y, w) */
    double *score;
    int32_t *prev;
    ChainNode *tree;
    int32_t *nEnt; /* taking-part triples */
};

__device__ __forceinline__ ChainWork chain_work(char *base, int64_t m, int64_t lX, int64_t lY) {
    ChainWork w;
    w.count = reinterpret_cast<int32_t *>(base);
    base += dec_round(4 * (lX + 1));
    w.ent = reinterpret_cast<int3 *>(base);
    base += dec_round(12 * m);
    w.score = reinterpret_cast<double *>(base);
    base += dec_round(8 * m);
    w.prev = reinterpret_cast<int32_t *>(base);
    base += dec_round(4 * m);
    w.tree = reinterpret_cast<ChainNode *>(base);
    base += dec_round(16 * (lY + 1));
    w.nEnt = reinterpret_cast<int32_t *>(base);
    return w;
}

/* chain_better of realign.c: higher score, then smaller y, then the later triple of the (x ascending, y descending) order -- a total
 * order on chain ends, so a maximum over any set of nodes does not depend on the order it is taken in */
__device__ __forceinline__ bool chain_node_better(const ChainNode &a, const ChainNode &b) {
    if (b.idx < 0) return a.idx >= 0;
    if (a.idx < 0) return false;
    if (a.score != b.score) return a.score > b.score;
    if (a.y != b.y) return a.y < b.y;
    return a.idx > b.idx;
}

__device__ __forceinline__ ChainNode chain_warp_max(ChainNode v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ChainNode u;
        u.score = __shfl_xor_sync(0xFFFFFFFFu, v.score, o);
        u.y = __shfl_xor_sync(0xFFFFFFFFu, v.y, o);
        u.idx = __shfl_xor_sync(0xFFFFFFFFu, v.idx, o);
        if (chain_node_better(u, v)) v = u;
    }
    return v;
}

__device__ __forceinline__ bool chain_takes_part(int32_t w, double matchGamma) {
    const double d = (double) w / CPB_PAIR_ALIGNMENT_PROB_1;
    return d >= matchGamma && d > 0.0;
}

/* One warp per pair: counting sort of the taking-part triples by x, y descending inside an x.  The device list is ordered by (x + y, x),
 * so the triples of one x come in y ascending: each takes the highest free slot of its bucket, in list order. */
__global__ void k_chain_sort(const DecodePair *P, int nP, const int32_t *list0, char *scratch, double matchGamma) {
    const int pi = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pi >= nP) return;
    const DecodePair D = P[pi];
    ChainWork W = chain_work(scratch + D.work, D.n0, D.lX, D.lY);
    for (int64_t x = lane; x <= D.lX; x += 32) W.count[x] = 0;
    __syncwarp();
    const int32_t *t = list0 + 3 * D.list0;
    for (int64_t k = lane; k < D.n0; k += 32) {
        if (chain_takes_part(t[3 * k], matchGamma)) atomicAdd(&W.count[t[3 * k + 1]], 1);
    }
    __syncwarp();
    /* inclusive scan: count[x] becomes the end of bucket x */
    int32_t carry = 0;
    for (int64_t x0 = 0; x0 <= D.lX; x0 += 32) {
        const int64_t x = x0 + lane;
        int32_t v = x <= D.lX ? W.count[x] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int32_t u = __shfl_up_sync(0xFFFFFFFFu, v, o);
            if (lane >= o) v += u;
        }
        if (x <= D.lX) W.count[x] = carry + v;
        carry += __shfl_sync(0xFFFFFFFFu, v, 31);
    }
    if (lane == 0) *W.nEnt = carry;
    __syncwarp();
    for (int64_t k0 = 0; k0 < D.n0; k0 += 32) {
        const int64_t k = k0 + lane;
        const bool in = k < D.n0 && chain_takes_part(t[3 * k], matchGamma);
        const int32_t x = in ? t[3 * k + 1] : -1 - lane;
        const unsigned peers = __match_any_sync(0xFFFFFFFFu, x);
        int32_t end = 0;
        if (in) end = W.count[x];
        __syncwarp();
        if (in) {
            const int rank = __popc(peers & ((1u << lane) - 1));
            W.ent[end - 1 - rank] = make_int3(x, t[3 * k + 2], t[3 * k]);
            if ((peers >> lane) == 1u) W.count[x] = end - __popc(peers); /* the last lane of the group moves the bucket's end */
        }
        __syncwarp();
    }
}

/* One warp per pair: the host's sweep over x with a prefix-maximum tree over y.  The nodes of a prefix query [0, y) are y with its lowest
 * set bits cleared one by one, those of an update from y + 1 up the tree: lane l takes the l-th, all load at once and a shuffle reduction
 * takes the best.  All triples of one x look up before any of them is inserted.  lens[pi] and best[pi] receive the chain's length and
 * its last triple. */
__global__ void k_chain_sweep(const DecodePair *P, int nP, char *scratch, int32_t *lens, int32_t *best) {
    const int pi = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pi >= nP) return;
    const DecodePair D = P[pi];
    ChainWork W = chain_work(scratch + D.work, D.n0, D.lX, D.lY);
    const int lY = D.lY;
    for (int f = lane; f <= lY; f += 32) W.tree[f] = ChainNode{ 0.0, 0, -1 };
    __syncwarp();
    const int m = *W.nEnt;
    ChainNode top{ 0.0, 0, -1 };
    for (int i = 0; i < m;) {
        const int x = W.ent[i].x;
        int j = i;
        while (j < m && W.ent[j].x == x) j++;
        for (int k = i; k < j; k++) {
            const int3 e = W.ent[k];
            int f = e.y;
            for (int s = 0; s < lane && f > 0; s++) f &= f - 1;
            ChainNode v{ 0.0, 0, -1 };
            if (f > 0) v = W.tree[f];
            v = chain_warp_max(v);
            if (lane == 0) {
                W.prev[k] = v.idx;
                W.score[k] = (v.idx >= 0 ? v.score : 0.0) + (double) e.z / CPB_PAIR_ALIGNMENT_PROB_1;
            }
        }
        __syncwarp();
        for (int k = i; k < j; k++) { /* y descending, as the host inserts them */
            const ChainNode c{ W.score[k], W.ent[k].y, k };
            int64_t f = (int64_t) c.y + 1;
            for (int s = 0; s < lane && f <= lY; s++) f += f & -f;
            if (f <= lY && chain_node_better(c, W.tree[f])) W.tree[f] = c;
            if (chain_node_better(c, top)) top = c;
            __syncwarp();
        }
        i = j;
    }
    if (lane == 0) {
        int len = 0;
        for (int k = top.idx; k >= 0; k = W.prev[k]) len++;
        lens[pi] = len;
        best[pi] = top.idx;
    }
}

/* the chain, first triple first, at out[off[pi]] */
__global__ void k_chain_write(const DecodePair *P, int nP, char *scratch, const int32_t *lens, const int32_t *best, const int64_t *off, int32_t *out) {
    const int pi = blockIdx.x * blockDim.x + threadIdx.x;
    if (pi >= nP) return;
    const DecodePair D = P[pi];
    ChainWork W = chain_work(scratch + D.work, D.n0, D.lX, D.lY);
    int64_t at = off[pi] + lens[pi];
    for (int k = best[pi]; k >= 0; k = W.prev[k]) {
        at--;
        const int3 e = W.ent[k];
        out[3 * at] = e.z;
        out[3 * at + 1] = e.x;
        out[3 * at + 2] = e.y;
    }
}

/* ---- maximal expected accuracy ----
 * Work arrays of a pair with m triples in list 0: list 0 in the reference's order, the DP's scores, back pointers and isHigh flags
 * (m + 1 entries: the last is the virtual pair at (lX, lY)), the cumulative gap weights of X and Y, and the least (x, y) of every aligned
 * chunk of 32 and block of 1024 reference-ordered triples (k_mea_summaries; what lets k_mea skip ranges that hold no predecessor). */
__host__ __device__ __forceinline__ int64_t mea_chunks(int64_t m) { return (m + 31) >> 5; }
__host__ __device__ __forceinline__ int64_t mea_blocks(int64_t m) { return (mea_chunks(m) + 31) >> 5; }

__host__ __device__ __forceinline__ int64_t mea_work_bytes(int64_t m, int64_t lX, int64_t lY) {
    return dec_round(12 * m) + dec_round(8 * (m + 1)) + dec_round(4 * (m + 1)) + dec_round(m + 1) + dec_round(8 * lX) + dec_round(8 * lY) +
           dec_round(8 * mea_chunks(m)) + dec_round(8 * mea_blocks(m));
}

struct MeaWork {
    int3 *ref; /* (pInt, x, y) */
    double *score;
    int32_t *back;
    uint8_t *high;
    long long *cumX, *cumY;
    int2 *chunk, *block; /* least (x, y) of triples 32c ... 32c + 31, and of 1024b ... 1024b + 1023 */
};

__device__ __forceinline__ MeaWork mea_work(char *base, int64_t m, int64_t lX, int64_t lY) {
    MeaWork w;
    w.ref = reinterpret_cast<int3 *>(base);
    base += dec_round(12 * m);
    w.score = reinterpret_cast<double *>(base);
    base += dec_round(8 * (m + 1));
    w.back = reinterpret_cast<int32_t *>(base);
    base += dec_round(4 * (m + 1));
    w.high = reinterpret_cast<uint8_t *>(base);
    base += dec_round(m + 1);
    w.cumX = reinterpret_cast<long long *>(base);
    base += dec_round(8 * lX);
    w.cumY = reinterpret_cast<long long *>(base);
    base += dec_round(8 * lY);
    w.chunk = reinterpret_cast<int2 *>(base);
    base += dec_round(8 * mea_chunks(m));
    w.block = reinterpret_cast<int2 *>(base);
    return w;
}

/* One thread per pair: list 0 of the pair in the order libcpecan.so hands it over (regions ascending; inside a region the traceback blocks
 * last to first; inside a block x + y ascending and x descending), the permutation cpb_batch_fetch_pairs_reference_order makes on the host.
 * Block j of region r owns the diagonals up to blockFrom[regBlock0[r] + j] + regShift[r]; triples after the pair's last block keep
 * their place. */
__global__ void k_ref_order(const DecodePair *P, int nP, const int32_t *list0, const int64_t *regShift, const int64_t *regBlock0,
                            const int32_t *regBlocks, const int32_t *blockFrom, char *scratch) {
    const int pi = blockIdx.x * blockDim.x + threadIdx.x;
    if (pi >= nP) return;
    const DecodePair D = P[pi];
    MeaWork W = mea_work(scratch + D.work, D.n0, D.lX, D.lY);
    const int32_t *t = list0 + 3 * D.list0;
    const int64_t m = D.n0;
    int64_t cur = 0;
    for (int64_t r = D.region0; r < D.region1; r++) {
        const int64_t shift = regShift[r], b0 = regBlock0[r];
        const int nb = regBlocks[r];
        const int64_t first = cur;
        for (int j = 0; j < nb; j++) { /* the region's end */
            const int64_t hi = (int64_t) blockFrom[b0 + j] + shift;
            while (cur < m && (int64_t) t[3 * cur + 1] + t[3 * cur + 2] <= hi) cur++;
        }
        const int64_t last = cur;
        int64_t a = first;
        for (int j = 0; j < nb; j++) {
            const int64_t hi = (int64_t) blockFrom[b0 + j] + shift;
            int64_t e = a;
            while (e < m && (int64_t) t[3 * e + 1] + t[3 * e + 2] <= hi) e++;
            const int64_t base = first + (last - e); /* the blocks after this one come first */
            for (int64_t g0 = a; g0 < e;) {
                const int64_t sum = (int64_t) t[3 * g0 + 1] + t[3 * g0 + 2];
                int64_t g1 = g0 + 1;
                while (g1 < e && (int64_t) t[3 * g1 + 1] + t[3 * g1 + 2] == sum) g1++;
                for (int64_t k = g0; k < g1; k++) W.ref[base + (g0 - a) + (g1 - 1 - k)] = make_int3(t[3 * k], t[3 * k + 1], t[3 * k + 2]);
                g0 = g1;
            }
            a = e;
        }
    }
    for (; cur < m; cur++) W.ref[cur] = make_int3(t[3 * cur], t[3 * cur + 1], t[3 * cur + 2]);
}

/* One thread per pair, after k_ref_order: with out == nullptr the pair's list length to lens[pi]; otherwise its reference-ordered list to
 * out[off[pi]...] (the test-support path that compares the permutation with cpb_batch_fetch_pairs_reference_order) */
__global__ void k_ref_emit(const DecodePair *P, int nP, char *scratch, int32_t *lens, const int64_t *off, int32_t *out) {
    const int pi = blockIdx.x * blockDim.x + threadIdx.x;
    if (pi >= nP) return;
    const DecodePair D = P[pi];
    if (out == nullptr) {
        lens[pi] = D.n0;
        return;
    }
    MeaWork W = mea_work(scratch + D.work, D.n0, D.lX, D.lY);
    for (int64_t k = 0; k < D.n0; k++) {
        const int3 e = W.ref[k];
        out[3 * (off[pi] + k)] = e.x;
        out[3 * (off[pi] + k) + 1] = e.y;
        out[3 * (off[pi] + k) + 2] = e.z;
    }
}

/* One warp per pair: cumX[i] = the gap-X weights of positions 0..i (list 1 by x), cumY likewise (list 2 by y) */
__global__ void k_mea_gaps(const DecodePair *P, int nP, const int32_t *list1, const int32_t *list2, char *scratch) {
    const int pi = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pi >= nP) return;
    const DecodePair D = P[pi];
    MeaWork W = mea_work(scratch + D.work, D.n0, D.lX, D.lY);
    for (int side = 0; side < 2; side++) {
        long long *cum = side == 0 ? W.cumX : W.cumY;
        const int64_t len = side == 0 ? D.lX : D.lY;
        const int32_t *t = side == 0 ? list1 + 3 * D.gap1 : list2 + 3 * D.gap2;
        const int64_t n = side == 0 ? D.n1 : D.n2;
        const int field = side == 0 ? 1 : 2;
        for (int64_t i = lane; i < len; i += 32) cum[i] = 0;
        __syncwarp();
        for (int64_t k = lane; k < n; k += 32)
            atomicAdd(reinterpret_cast<unsigned long long *>(cum + t[3 * k + field]), (unsigned long long) (long long) t[3 * k]);
        __syncwarp();
        long long carry = 0;
        for (int64_t i0 = 0; i0 < len; i0 += 32) {
            const int64_t i = i0 + lane;
            long long v = i < len ? cum[i] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long u = __shfl_up_sync(0xFFFFFFFFu, v, o);
                if (lane >= o) v += u;
            }
            if (i < len) cum[i] = carry + v;
            carry += __shfl_sync(0xFFFFFFFFu, v, 31);
        }
        __syncwarp();
    }
}

__device__ __forceinline__ int2 mea_least(int2 v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v.x = min(v.x, __shfl_xor_sync(0xFFFFFFFFu, v.x, o));
        v.y = min(v.y, __shfl_xor_sync(0xFFFFFFFFu, v.y, o));
    }
    return v;
}

/* One warp per pair, after k_ref_order: the least (x, y) of every chunk of 32 reference-ordered triples, then of every block of 32 chunks */
__global__ void k_mea_summaries(const DecodePair *P, int nP, char *scratch) {
    const int pi = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pi >= nP) return;
    const DecodePair D = P[pi];
    MeaWork W = mea_work(scratch + D.work, D.n0, D.lX, D.lY);
    const int m = D.n0, nChunks = (int) mea_chunks(m), nBlocks = (int) mea_blocks(m);
    for (int c = 0; c < nChunks; c++) {
        const int j = (c << 5) + lane;
        const int2 v = mea_least(j < m ? make_int2(W.ref[j].y, W.ref[j].z) : make_int2(INT32_MAX, INT32_MAX));
        if (lane == 0) W.chunk[c] = v;
    }
    __syncwarp();
    for (int b = 0; b < nBlocks; b++) {
        const int c = (b << 5) + lane;
        const int2 v = mea_least(c < nChunks ? W.chunk[c] : make_int2(INT32_MAX, INT32_MAX));
        if (lane == 0) W.block[b] = v;
    }
}

/* may the triples a summary covers hold a predecessor of (x, y)? */
__device__ __forceinline__ bool mea_may_precede(int2 least, int64_t x, int64_t y) { return least.x < x && least.y < y; }

/* The highest chunk at or below c that may hold a predecessor of (x, y), or -1; the same on every lane.  A chunk whose least x or least y
 * is not below the pair's holds none, and its triples would all be passed over by the scan.  The chunk c itself is tried first (the common
 * case inside a block: one broadcast load).  Then the lanes test the 32 block summaries of c's group of 32 blocks (the blocks above c's
 * excluded), and the highest block that may hold one has its 32 chunk summaries tested at once (the chunks above c excluded); a group or a
 * block without a hit is passed whole, so the walk over the later blocks of a region costs one step per 32 768 triples. */
__device__ __forceinline__ int mea_next_chunk(const MeaWork &W, int c, int64_t x, int64_t y, int lane) {
    if (c < 0) return -1;
    if (mea_may_precede(W.chunk[c], x, y)) return c;
    c--;
    while (c >= 0) {
        const int b = c >> 5, g = b & ~31;
        unsigned hit = __ballot_sync(0xFFFFFFFFu, g + lane <= b && mea_may_precede(W.block[g + lane], x, y));
        if (hit == 0) {
            c = (g << 5) - 1;
            continue;
        }
        const int hb = g + 31 - __clz(hit);
        if (hb < b) c = (hb << 5) + 31;
        const int k = hb << 5;
        hit = __ballot_sync(0xFFFFFFFFu, k + lane <= c && mea_may_precede(W.chunk[k + lane], x, y));
        if (hit != 0) return k + 31 - __clz(hit);
        c = k - 1;
    }
    return -1;
}

/* gap_weight of realign.c: the weights of positions start .. start + length - 1 */
__device__ __forceinline__ long long mea_gap(const long long *cum, int64_t start, int64_t length) {
    return length == 0 ? 0 : cum[start + length - 1] - (start > 0 ? cum[start - 1] : 0);
}

/* (int64 gap weight) * (float gamma), in float as C evaluates it */
__device__ __forceinline__ float mea_gap_term(long long g, float gamma) { return __fmul_rn(__ll2float_rn(g), gamma); }

/* One warp per pair: the DP of getMaximalExpectedAccuracyPairwiseAlignment over the reference-ordered list, sequential in i.  For pair i
 * the host scans j = i-1, i-2, ... keeping the first strictly larger truncated candidate among the valid predecessors (x2 < x, y2 < y),
 * and stops after the first valid one with isHigh set.  Here the warp takes the aligned chunks of 32 triples from the one holding i - 1
 * down, lane l the triple 32c + 31 - l (those at or above i are not valid), and skips every chunk that holds no valid predecessor
 * (mea_next_chunk): such a chunk changes nothing in the scan.  In a loaded chunk the cutoff is the nearest valid isHigh lane (included),
 * and the maximum over valid lanes up to it by (candidate larger, then j larger) is what the strict-> scan selects; it replaces the running
 * score only if strictly larger.  scores[pi] receives maxScore, lens[pi] the length of the traceback. */
__global__ void k_mea(const DecodePair *P, int nP, char *scratch, float gamma, double *scores, int32_t *lens) {
    const int pi = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pi >= nP) return;
    const DecodePair D = P[pi];
    MeaWork W = mea_work(scratch + D.work, D.n0, D.lX, D.lY);
    const int m = D.n0;
    const int64_t lX = D.lX, lY = D.lY;
    double maxScore = 0;
    for (int i = 0; i <= m; i++) {
        long long w = 0;
        int64_t x = lX, y = lY;
        if (i < m) {
            const int3 e = W.ref[i];
            w = e.x;
            x = e.y;
            y = e.z;
        }
        /* w + (gx + gy) * gamma: all float, then widened */
        double score = (double) __fadd_rn(__ll2float_rn(w), mea_gap_term(mea_gap(W.cumX, 0, x) + mea_gap(W.cumY, 0, y), gamma));
        int from = -1;
        for (int c = mea_next_chunk(W, i > 0 ? (i - 1) >> 5 : -1, x, y, lane); c >= 0; c = mea_next_chunk(W, c - 1, x, y, lane)) {
            const int j = (c << 5) + 31 - lane;
            bool valid = false, isHigh = false;
            double s = 0.0;
            if (j < i) {
                const int3 q = W.ref[j];
                const int64_t x2 = q.y, y2 = q.z;
                if (x2 < x && y2 < y) {
                    valid = true;
                    isHigh = W.high[j] != 0;
                    /* (int64) (w + scores[j] + (gap) * gamma): double, the gap term in float, then truncated */
                    const double c = __dadd_rn(__dadd_rn((double) w, W.score[j]),
                                               (double) mea_gap_term(mea_gap(W.cumX, x2 + 1, x - x2 - 1) + mea_gap(W.cumY, y2 + 1, y - y2 - 1), gamma));
                    s = (double) (long long) c;
                }
            }
            const unsigned highs = __ballot_sync(0xFFFFFFFFu, isHigh);
            if (highs != 0 && lane > __ffs(highs) - 1) valid = false;
            double bs = valid ? s : -INFINITY;
            int bj = valid ? j : -1;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double os = __shfl_xor_sync(0xFFFFFFFFu, bs, o);
                const int oj = __shfl_xor_sync(0xFFFFFFFFu, bj, o);
                if (oj >= 0 && (bj < 0 || os > bs || (os == bs && oj > bj))) {
                    bs = os;
                    bj = oj;
                }
            }
            if (bj >= 0 && bs > score) {
                score = bs;
                from = bj;
            }
            if (highs != 0) break;
        }
        const int64_t tX = x < lX ? mea_gap(W.cumX, x + 1, lX - x - 1) : 0, tY = y < lY ? mea_gap(W.cumY, y + 1, lY - y - 1) : 0;
        const double s = __dadd_rn(score, (double) mea_gap_term(tX + tY, gamma));
        const bool high = s >= maxScore;
        if (high) maxScore = s;
        if (lane == 0) {
            W.back[i] = from;
            W.score[i] = score;
            W.high[i] = high;
        }
        __syncwarp();
    }
    if (lane == 0) {
        int len = 0;
        for (int k = W.back[m]; k >= 0; k = W.back[k]) len++;
        scores[pi] = maxScore;
        lens[pi] = len;
    }
}

/* One thread per pair, after k_mea: the MEA alignment (SHIFT false), or leftShiftAlignment of it (SHIFT true), walking the traceback
 * from its last pair as the host walks the list from its end.  With out == nullptr only the length goes to lens[pi]; otherwise the
 * triples go to out[off[pi]...], first pair first.  X and Y are the kept upper-cased bytes. */
template <bool SHIFT>
__global__ void k_decode_emit(const DecodePair *P, int nP, char *scratch, const uint8_t *X, const uint8_t *Y, int32_t *lens, const int64_t *off,
                              int32_t *out) {
    const int pi = blockIdx.x * blockDim.x + threadIdx.x;
    if (pi >= nP) return;
    const DecodePair D = P[pi];
    MeaWork W = mea_work(scratch + D.work, D.n0, D.lX, D.lY);
    const uint8_t *sx = X + D.seqX, *sy = Y + D.seqY;
    int64_t appended = 0;
    const int64_t len = out != nullptr ? off[pi + 1] - off[pi] : 0;
    auto emit = [&](int32_t w, int64_t x, int64_t y) {
        if (out != nullptr) {
            const int64_t at = off[pi] + len - 1 - appended;
            out[3 * at] = w;
            out[3 * at + 1] = (int32_t) x;
            out[3 * at + 2] = (int32_t) y;
        }
        appended++;
    };
    if (!SHIFT) {
        for (int k = W.back[D.n0]; k >= 0; k = W.back[k]) emit(W.ref[k].x, W.ref[k].y, W.ref[k].z);
    } else {
        int64_t x = D.lX, y = D.lY;
        int32_t firstW = 1; /* the weight of the alignment's first pair, 1 if it has none */
        for (int k = W.back[D.n0]; k >= 0; k = W.back[k]) {
            const int3 e = W.ref[k];
            const int32_t w = e.x;
            const int64_t x2 = e.y, y2 = e.z;
            firstW = w;
            while ((x - x2 > 1 || y - y2 > 1) && sx[x - 1] == sy[y - 1]) {
                emit(w, x - 1, y - 1);
                x--;
                y--;
                if (x2 == x || y2 == y) break;
            }
            if (x2 < x && y2 < y) {
                emit(w, x2, y2);
                x = x2;
                y = y2;
            }
        }
        while (x > 0 && y > 0 && sx[x - 1] == sy[y - 1]) {
            emit(firstW, x - 1, y - 1);
            x--;
            y--;
        }
    }
    if (out == nullptr) lens[pi] = (int32_t) appended;
}

/* ---- scores of the alignment list: one warp per pair ---- */
__global__ void k_decode_scores(const int32_t *aln, const int64_t *off, int nPairs, const int64_t *xOff, const int64_t *yOff, const uint8_t *X,
                                const uint8_t *Y, int kind, double *scores) {
    const int pair = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pair >= nPairs) return;
    const uint8_t *sx = X + xOff[pair], *sy = Y + yOff[pair];
    long long matches = 0, weight = 0;
    for (int64_t t = off[pair] + lane; t < off[pair + 1]; t += 32) {
        weight += aln[3 * t];
        const uint8_t cx = sx[aln[3 * t + 1]], cy = sy[aln[3 * t + 2]];
        matches += cx == cy && cx != 'N';
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        matches += __shfl_xor_sync(0xFFFFFFFFu, matches, o);
        weight += __shfl_xor_sync(0xFFFFFFFFu, weight, o);
    }
    if (lane != 0) return;
    const int64_t lXY = (xOff[pair + 1] - xOff[pair]) + (yOff[pair + 1] - yOff[pair]), len = off[pair + 1] - off[pair];
    /* the host sums the weights in double one by one: every partial sum is an integer below 2^53, so this is the same number */
    const double total = (double) weight;
    double s;
    switch (kind) {
    case CPB_SCORE_IDENTITY:
        s = 100.0 * (lXY == 0 ? 0.0 : __ddiv_rn(2.0 * (double) matches, (double) lXY));
        break;
    case CPB_SCORE_IDENTITY_IGNORING_GAPS:
        s = __ddiv_rn(100.0 * (double) matches, (double) len);
        break;
    case CPB_SCORE_POSTERIOR:
        s = 100.0 * (lXY == 0 ? 0.0 : __ddiv_rn(2.0 * total, (double) (lXY * (int64_t) CPB_PAIR_ALIGNMENT_PROB_1)));
        break;
    default:
        s = __ddiv_rn(100.0 * total, (double) len * (double) CPB_PAIR_ALIGNMENT_PROB_1);
        break;
    }
    scores[pair] = s;
}

/* ---- anchors from the alignment list (cpb_batch_anchors_from_alignments) ----
 * The anchors job_prepare (host/realignJobs.h) builds from the cigar cPecanRealign writes for an alignment (pairs_to_alignment): the cigar's
 * match operations are the alignment's maximal diagonal runs (each next pair at (x + 1, y + 1)); convertPairwiseForwardStrandAlignmentToAnchorPairs
 * (realign.c:32-72) takes the columns at positions l in [trim, L - trim) of a run of length L, i.e. those with at least trim pairs of their
 * run before and after them; columns_match keeps those whose two bytes are equal and not N.  DecodePair.list0 / n0 say where a pair's
 * alignment is.  Work array of a pair of m triples: per triple the number of its run's triples before it, then its keep flag. */
__host__ __device__ __forceinline__ int64_t reanchor_work_bytes(int64_t m) { return dec_round(4 * m); }

/* columns_match of host/realignJobs.h on the kept bytes, which are already upper-cased: a column constrains the band iff its two bytes are
 * equal and not N */
__device__ __forceinline__ bool columns_match(uint8_t cx, uint8_t cy) { return cx == cy && cx != 'N'; }

/* One warp per pair, O(1) per triple: a forward sweep finds every triple's run start (the last start at or before it: the chunk's ballot,
 * or the run carried in from the chunks before), a backward sweep its run end likewise; lens[pi] receives the number of kept columns. */
__global__ void k_reanchor_count(const DecodePair *P, int nP, const int32_t *aln, const uint8_t *X, const uint8_t *Y, char *scratch, int32_t trim,
                                 int32_t *lens) {
    const int pi = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pi >= nP) return;
    const DecodePair D = P[pi];
    const int32_t *t = aln + 3 * D.list0;
    int32_t *w = reinterpret_cast<int32_t *>(scratch + D.work);
    const int m = D.n0;
    auto diagonal = [&](int k) { return t[3 * k + 1] == t[3 * k - 2] + 1 && t[3 * k + 2] == t[3 * k - 1] + 1; }; /* triple k follows k - 1 */
    int carry = 0;
    for (int k0 = 0; k0 < m; k0 += 32) {
        const int k = k0 + lane;
        const unsigned starts = __ballot_sync(0xFFFFFFFFu, k < m && (k == 0 || !diagonal(k)));
        const unsigned upTo = starts & (0xFFFFFFFFu >> (31 - lane));
        if (k < m) w[k] = k - (upTo != 0 ? k0 + 31 - __clz(upTo) : carry);
        if (starts != 0) carry = k0 + 31 - __clz(starts);
    }
    __syncwarp();
    const uint8_t *sx = X + D.seqX, *sy = Y + D.seqY;
    int kept = 0;
    carry = m - 1;
    for (int k0 = (m - 1) & ~31; k0 >= 0; k0 -= 32) {
        const int k = k0 + lane;
        const unsigned ends = __ballot_sync(0xFFFFFFFFu, k < m && (k == m - 1 || !diagonal(k + 1)));
        const unsigned from = ends & (0xFFFFFFFFu << lane);
        bool keep = false;
        if (k < m) {
            const int end = from != 0 ? k0 + __ffs(from) - 1 : carry;
            const uint8_t cx = sx[t[3 * k + 1]], cy = sy[t[3 * k + 2]];
            keep = w[k] >= trim && end - k >= trim && columns_match(cx, cy);
            w[k] = keep;
        }
        kept += __popc(__ballot_sync(0xFFFFFFFFu, keep));
        if (ends != 0) carry = k0 + __ffs(ends) - 1;
    }
    if (lane == 0) lens[pi] = kept;
}

/* One warp per pair, after the scan of lens: the kept columns as (x, y, expansion) at out[off[pi]...], x ascending */
__global__ void k_reanchor_write(const DecodePair *P, int nP, const int32_t *aln, const char *scratch, int32_t expansion, const int64_t *off, int32_t *out) {
    const int pi = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pi >= nP) return;
    const DecodePair D = P[pi];
    const int32_t *t = aln + 3 * D.list0;
    const int32_t *w = reinterpret_cast<const int32_t *>(scratch + D.work);
    int64_t at = off[pi];
    for (int k0 = 0; k0 < D.n0; k0 += 32) {
        const int k = k0 + lane;
        const bool keep = k < D.n0 && w[k] != 0;
        const unsigned keeps = __ballot_sync(0xFFFFFFFFu, keep);
        if (keep) {
            const int64_t o = at + __popc(keeps & ((1u << lane) - 1));
            out[3 * o] = t[3 * k + 1];
            out[3 * o + 1] = t[3 * k + 2];
            out[3 * o + 2] = expansion;
        }
        at += __popc(keeps);
    }
}

/* ---- cigar operations of the alignment list (cpb_batch_alignment_cigars) ----
 * pairs_to_alignment of cPecanRealign.c:98-123 for every pair: before column k an INDEL_X of x_k - x_{k-1} - 1 and an INDEL_Y of
 * y_k - y_{k-1} - 1 where positive, with (x_-1, y_-1) = (-1, -1); then the column, which starts a MATCH operation if it is the first or
 * follows a gap; after the last column an INDEL_X and an INDEL_Y up to (lX, lY).  A MATCH runs from its start column to the next start.
 * One warp per pair, 32 columns per step, no work array: every lane takes its predecessor by shuffle, lane 0 from memory. */
__device__ __forceinline__ void cigar_column(const int32_t *t, int m, int k0, int lane, int32_t &gx, int32_t &gy, bool &start) {
    const int k = k0 + lane;
    int32_t x = 0, y = 0;
    if (k < m) {
        x = t[3 * k + 1];
        y = t[3 * k + 2];
    }
    int32_t px = __shfl_up_sync(0xFFFFFFFFu, x, 1), py = __shfl_up_sync(0xFFFFFFFFu, y, 1);
    if (lane == 0) {
        px = k0 > 0 ? t[3 * k0 - 2] : -1;
        py = k0 > 0 ? t[3 * k0 - 1] : -1;
    }
    gx = k < m ? x - px - 1 : 0;
    gy = k < m ? y - py - 1 : 0;
    start = k < m && (k == 0 || gx > 0 || gy > 0);
}

/* the trailing INDEL_X and INDEL_Y of a pair of m columns */
__device__ __forceinline__ void cigar_tail(const int32_t *t, int m, int64_t lX, int64_t lY, int32_t &tx, int32_t &ty) {
    tx = (int32_t) (lX - (m > 0 ? t[3 * m - 2] : -1) - 1);
    ty = (int32_t) (lY - (m > 0 ? t[3 * m - 1] : -1) - 1);
}

/* lens[pair] = the number of operations of the pair's cigar (at most 3m + 2) */
__global__ void k_cigar_count(const int32_t *aln, const int64_t *off, int nPairs, const int64_t *xOff, const int64_t *yOff, int32_t *lens) {
    const int pair = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pair >= nPairs) return;
    const int32_t *t = aln + 3 * off[pair];
    const int m = (int) (off[pair + 1] - off[pair]);
    int32_t count = 0, gx, gy;
    bool start;
    for (int k0 = 0; k0 < m; k0 += 32) {
        cigar_column(t, m, k0, lane, gx, gy, start);
        count += (gx > 0) + (gy > 0) + start;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) count += __shfl_xor_sync(0xFFFFFFFFu, count, o);
    if (lane != 0) return;
    int32_t tx, ty;
    cigar_tail(t, m, xOff[pair + 1] - xOff[pair], yOff[pair + 1] - yOff[pair], tx, ty);
    lens[pair] = count + (tx > 0) + (ty > 0);
}

/* After the scan of lens: the pair's operations as int32 (type, length) at ops[2 * opOff[pair]...].  The steps run last to first, so the
 * next MATCH start after a lane's is the next start bit of the step's ballot or, if there is none, the first start of the steps after it
 * (m past the last run); each lane's first operation is the step's end minus the operations of the lanes from it to 31. */
__global__ void k_cigar_write(const int32_t *aln, const int64_t *off, int nPairs, const int64_t *xOff, const int64_t *yOff, const int64_t *opOff,
                              int32_t *ops) {
    const int pair = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pair >= nPairs) return;
    const int32_t *t = aln + 3 * off[pair];
    const int m = (int) (off[pair + 1] - off[pair]);
    int2 *out = reinterpret_cast<int2 *>(ops);
    int32_t tx, ty;
    cigar_tail(t, m, xOff[pair + 1] - xOff[pair], yOff[pair + 1] - yOff[pair], tx, ty);
    int64_t at = opOff[pair + 1] - (tx > 0) - (ty > 0); /* one past the operation of the last column */
    if (lane == 0) {
        if (tx > 0) out[at] = make_int2(CPB_OP_INDEL_X, tx);
        if (ty > 0) out[at + (tx > 0)] = make_int2(CPB_OP_INDEL_Y, ty);
    }
    int32_t next = m, gx, gy;
    bool start;
    for (int k0 = (m - 1) & ~31; k0 >= 0; k0 -= 32) {
        cigar_column(t, m, k0, lane, gx, gy, start);
        int32_t s = (gx > 0) + (gy > 0) + start; /* then: the operations of lanes lane..31 */
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int32_t u = __shfl_down_sync(0xFFFFFFFFu, s, o);
            if (lane + o < 32) s += u;
        }
        const unsigned starts = __ballot_sync(0xFFFFFFFFu, start), after = starts & (0xFFFFFFFEu << lane);
        int64_t w = at - s;
        if (gx > 0) out[w++] = make_int2(CPB_OP_INDEL_X, gx);
        if (gy > 0) out[w++] = make_int2(CPB_OP_INDEL_Y, gy);
        if (start) out[w] = make_int2(CPB_OP_MATCH, (after != 0 ? k0 + __ffs(after) - 1 : next) - (k0 + lane));
        at -= __shfl_sync(0xFFFFFFFFu, s, 0);
        if (starts != 0) next = k0 + __ffs(starts) - 1;
    }
}

/* ---- alignments given as cigar operations (cpb_batch_create_from_cigars, cpb_batch_alignments_from_cigars) ----
 * A pair's operations, int32 (type, length) at ops[2 * opOff[pair]...], walk from (0, 0) to (lX, lY); the host has checked that they do.
 * A MATCH of length L at (x, y) gives the columns (x + l, y + l) for l in [trim, L - trim), adjacent MATCH operations each trimmed
 * (convertPairwiseForwardStrandAlignmentToAnchorPairs, realign.c:32-72).  One warp per pair, 32 operations per step, no work array:
 * warp scans of the x and y advances and of the column counts give every operation its start and its first column, carried across
 * steps; the step's columns are then dealt to the lanes 32 at a time, each lane finding its operation by a binary search over the
 * lanes' first columns.  O(1) per operation and per column.  cigar_columns calls f(t, valid, x, y) on every lane for the columns
 * t = t0 + lane of the step, counted from the pair's first column, and valid = false past the step's last. */
template <class F>
__device__ __forceinline__ void cigar_columns(const int32_t *ops, int64_t o0, int64_t o1, int32_t trim, int lane, F f) {
    int32_t x0 = 0, y0 = 0, c0 = 0; /* where the step's first operation starts, and its first column */
    for (int64_t k0 = o0; k0 < o1; k0 += 32) {
        const int64_t k = k0 + lane;
        int32_t type = CPB_OP_INDEL_X, len = 0;
        if (k < o1) {
            type = ops[2 * k];
            len = ops[2 * k + 1];
        }
        const int32_t dx = type != CPB_OP_INDEL_Y ? len : 0, dy = type != CPB_OP_INDEL_X ? len : 0;
        const int32_t c = type == CPB_OP_MATCH && (int64_t) len > 2 * (int64_t) trim ? len - 2 * trim : 0;
        int32_t sx = dx, sy = dy, sc = c; /* inclusive scans */
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int32_t ux = __shfl_up_sync(0xFFFFFFFFu, sx, o), uy = __shfl_up_sync(0xFFFFFFFFu, sy, o), uc = __shfl_up_sync(0xFFFFFFFFu, sc, o);
            if (lane >= o) {
                sx += ux;
                sy += uy;
                sc += uc;
            }
        }
        const int32_t x = x0 + sx - dx, y = y0 + sy - dy, first = sc - c; /* the operation's start, and its first column within the step */
        const int32_t total = __shfl_sync(0xFFFFFFFFu, sc, 31);
        for (int32_t t0 = 0; t0 < total; t0 += 32) {
            const int32_t t = t0 + lane;
            int lo = 0; /* the last operation whose first column is at or before t: one with columns when t < total */
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) {
                if (__shfl_sync(0xFFFFFFFFu, first, lo + s) <= t) lo += s;
            }
            const int32_t at = trim + (t - __shfl_sync(0xFFFFFFFFu, first, lo)); /* l of the column in its operation */
            f(c0 + t, t < total, __shfl_sync(0xFFFFFFFFu, x, lo) + at, __shfl_sync(0xFFFFFFFFu, y, lo) + at);
        }
        x0 += __shfl_sync(0xFFFFFFFFu, sx, 31);
        y0 += __shfl_sync(0xFFFFFFFFu, sy, 31);
        c0 += total;
    }
}

/* lens[pair] = the number of the pair's columns that columns_match keeps (the anchors job_prepare keeps) */
__global__ void k_cigar_cols_count(const int32_t *ops, const int64_t *opOff, int nPairs, const int64_t *xOff, const int64_t *yOff, const uint8_t *X,
                                   const uint8_t *Y, int32_t trim, int32_t *lens) {
    const int pair = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pair >= nPairs) return;
    const uint8_t *sx = X + xOff[pair], *sy = Y + yOff[pair];
    int32_t kept = 0;
    cigar_columns(ops, opOff[pair], opOff[pair + 1], trim, lane,
                  [&](int32_t, bool valid, int32_t x, int32_t y) { kept += __popc(__ballot_sync(0xFFFFFFFFu, valid && columns_match(sx[x], sy[y]))); });
    if (lane == 0) lens[pair] = kept;
}

/* After the scan: ANCHORS, the kept columns as (x, y, expansion) at out[off[pair]...]; otherwise every column as (0, x, y), the
 * alignment list before k_cigar_weigh.  x ascending. */
template <bool ANCHORS>
__global__ void k_cigar_cols_write(const int32_t *ops, const int64_t *opOff, int nPairs, const int64_t *xOff, const int64_t *yOff, const uint8_t *X,
                                   const uint8_t *Y, int32_t trim, int32_t expansion, const int64_t *off, int32_t *out) {
    const int pair = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pair >= nPairs) return;
    const uint8_t *sx = X + xOff[pair], *sy = Y + yOff[pair];
    int64_t at = off[pair];
    cigar_columns(ops, opOff[pair], opOff[pair + 1], trim, lane, [&](int32_t t, bool valid, int32_t x, int32_t y) {
        if (ANCHORS) {
            const bool keep = valid && columns_match(sx[x], sy[y]);
            const unsigned keeps = __ballot_sync(0xFFFFFFFFu, keep);
            if (keep) {
                const int64_t o = at + __popc(keeps & ((1u << lane) - 1));
                out[3 * o] = x;
                out[3 * o + 1] = y;
                out[3 * o + 2] = expansion;
            }
            at += __popc(keeps);
        } else if (valid) {
            out[3 * (at + t)] = 0;
            out[3 * (at + t) + 1] = x;
            out[3 * (at + t) + 2] = y;
        }
    });
}

/* One warp per pair, after k_cigar_cols_write<false>: every triple (w, x, y) of list 0 (l0Off: n+1 offsets) finds column x of the pair's
 * alignment by a binary search (the columns' x are strictly increasing) and, if that column is (x, y), gives it weight w.  (x, y) is
 * unique in list 0, so no two lanes write one column. */
__global__ void k_cigar_weigh(const int32_t *list0, const int64_t *l0Off, int nPairs, const int64_t *alnOff, int32_t *aln) {
    const int pair = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pair >= nPairs) return;
    int32_t *a = aln + 3 * alnOff[pair];
    const int64_t m = alnOff[pair + 1] - alnOff[pair];
    if (m == 0) return;
    for (int64_t k = l0Off[pair] + lane; k < l0Off[pair + 1]; k += 32) {
        const int32_t x = list0[3 * k + 1];
        int64_t lo = 0, hi = m; /* the first column with x at or above */
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (a[3 * mid + 1] < x) lo = mid + 1;
            else hi = mid;
        }
        if (lo < m && a[3 * lo + 1] == x && a[3 * lo + 2] == list0[3 * k + 2]) a[3 * lo] = list0[3 * k];
    }
}

} // namespace cpb
