/*
 * kernels.cuh -- sm_100a device code of the banded pair-HMM forward-backward.
 *
 * Data flow for one chunk of regions (a region = one split sub-problem, see engine.cu):
 *   k_band      per region : anchors -> per-diagonal band records + traceback-block schedule
 *   k_forward_strip  per region : anti-diagonal wavefront, one warp per region, lanes = matrix rows (strip_kernels.cuh);
 *                                 selected state planes (and full cells of "total" diagonals) -> HBM
 *   k_backward_strip per block  : same wavefront downwards in gather form; F + B planes (posterior modes) or
 *                                 B planes (expectations) -> HBM, per-cell F.B dot products of the total diagonals -> HBM
 *   k_totals    per decade : the reference's left-to-right logAdd folds that give totalProbability
 *   k_posterior per block  : exp(F+B-total) threshold scan, count pass then compacted write pass
 *   k_expect    per block  : expected transition / emission counts
 *
 * Arithmetic contract (bit-compatible with cPecan's C): all state is FP64, logAdd is the reference's
 * 4-segment cubic evaluated with separately rounded multiplies and adds (impl/pairwiseAligner.c:290-307),
 * every transition is from + (eP + tP) (:384,:394) and each cell accumulates its transitions in the
 * order the reference does (impl/stateMachine.c:454-479 / :695-713 forward; scatter order of
 * diagonalCalculationBackward re-expressed as a gather, SURVEY.md section 8a row a9).
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "cpecan_b200.h"

namespace cpb {

constexpr uint32_t NO_AUX = 0xFFFFFFFFu;
constexpr int XMY_BIAS = 1 << 30; /* even; makes xmy + bias positive so >>1 is a floor division */

struct __align__(16) DiagRec {
    int32_t xmyL;  /* smallest x-y on this diagonal */
    int32_t width; /* cells on this diagonal, (xmyR-xmyL)/2+1 */
    uint32_t coff; /* region-relative cell offset of the diagonal's first cell */
    uint32_t aoff; /* region-relative offset (in doubles) of the aux record if this is a "total" diagonal, else NO_AUX */
};

struct RegionDev {
    int64_t xBase, yBase;  /* first symbol of the region in the symbol arrays */
    int64_t anchorBase;    /* first anchor triple */
    int64_t diagBase;      /* first DiagRec; lX+lY+3 records (two sentinels) */
    int64_t blockBase;     /* first BlockRec slot */
    int64_t cellBase;      /* chunk-relative first cell (host, after planning) */
    int64_t auxBase;       /* chunk-relative first aux double (host, after planning) */
    int64_t maskBase;      /* chunk-relative first keep-mask word (host, after planning) */
    int64_t stripBase;     /* first StripRec of the region: (lX>>5)+1 records */
    int64_t cells;         /* out: band cells */
    int64_t auxDoubles;    /* out */
    int32_t lX, lY;
    int32_t nAnchors;
    int32_t pair;
    int32_t ox, oy;        /* region origin in pair coordinates */
    int32_t blockCap;
    int32_t nBlocks;       /* out */
    int32_t maxW;          /* out: widest diagonal */
    int32_t maxStripRange; /* out: longest diagonal range of a 32-row strip */
    int32_t err;           /* out: 0 ok, 1 invalid diagonal, 2 block table overflow */
    uint8_t raggedL, raggedR;
    uint8_t stripsSorted;  /* out: dFirst and dLast are non-decreasing along the strips (always, for a monotone band): block kernels
                            * then find their strips by bisection instead of scanning all of them */
    uint8_t pad_[5];
};

struct StripRec {
    int32_t dFirst, dLast; /* diagonals on which any row of the 32-row strip is inside the band (dLast < dFirst: never) */
};

/* bisection over the strips of a region with sorted strip records */
__device__ __forceinline__ int first_strip_with_last_at_least(const StripRec *strips, int n, int d) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (strips[mid].dLast >= d) hi = mid;
        else lo = mid + 1;
    }
    return lo; /* n if none */
}
__device__ __forceinline__ int last_strip_with_first_at_most(const StripRec *strips, int n, int d) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (strips[mid].dFirst <= d) lo = mid + 1;
        else hi = mid;
    }
    return lo - 1; /* -1 if none */
}

struct BlockRec {
    int32_t region;
    int32_t top;   /* diagonal the traceback starts from */
    int32_t T;     /* tracedBackTo before this block: owned diagonals are (T, from] */
    int32_t from;  /* tracedBackFrom */
    int32_t cells;   /* band cells on the diagonals (T, top] */
    int32_t atEnd;
    int64_t decadeBase; /* chunk-relative index of the block's first decade (host, after planning) */
    int64_t ckBase;     /* two-pass forward: offset (doubles) of the block's checkpoint, the full cells of diagonals T-1 and T */
};

/* Everything the DP kernels need besides the launch list. */
struct DpArgs {
    const RegionDev *regions;
    const BlockRec *blocks;
    const DiagRec *diags;
    const uint8_t *symX, *symY;
    double *planesF;       /* nPlanes planes of planeStride doubles */
    double *planesB;
    double *aux;
    double *totals;        /* per diagonal record (same indexing as diags) */
    int64_t planeStride;
    int32_t nPlanes;       /* 0 forward-only, 1 match, 3 match+gaps, S expectations */
    int32_t auxF;          /* planes of full forward state kept in aux records of total diagonals (S or 0) */
    const int32_t *list;   /* region ids (forward) or block ids (others) */
    double *forwardOut;    /* per region, forward-only mode */
    const double *ckpt;    /* two-pass forward: block checkpoints (k_forward_strip<..., FWD_BLOCKS>) */
};

/* ---------------------------------------------------------------------------------------------
 * logAdd, bit-compatible with impl/pairwiseAligner.c:290-307
 * ------------------------------------------------------------------------------------------- */
#ifndef CPB_TRUE_LOG_ZERO
#define CPB_FINITE_LOG_ZERO 1 /* default; -DCPB_TRUE_LOG_ZERO builds the kernels with -infinity as LOG_ZERO and the three-select logAdd */
#endif
/* the reference's 4-segment cubic, [segment][a,b,c,k]; the literals are floats promoted to double exactly as in C */
__constant__ double c_coefficients[16] = {
    (double) -0.009350833524763f, (double) 0.130659527668286f, (double) 0.498799810682272f, (double) 0.693203116424741f,
    (double) -0.014532321752540f, (double) 0.139942324101744f, (double) 0.495635523139337f, (double) 0.692140569840976f,
    (double) -0.004605031767994f, (double) 0.063427417320019f, (double) 0.695956496475118f, (double) 0.514272634594009f,
    (double) -0.000458661602210f, (double) 0.009695946122598f, (double) 0.930734667215156f, (double) 0.168037164329057f };

/*
 * Segment selection by table.  The segment bounds 1, 2.5 and 4.5 have a zero low word and a high word that is a
 * multiple of 2^17, so for d >= 0:  d > T  <=>  hi32(bits(d) - 1) >= hi32(T), and (hi32(bits(d) - 1) >> 17) - 0x1FF8
 * counts 2^17-wide buckets above 1.0.  A shared-memory table of LA_ROWS rows
 * maps the clamped bucket to its coefficients: rows 0-9: (1, 2.5]; rows 10-16: (2.5, 4.5]; rows 17-23: above 4.5 (the
 * polynomial is discarded from 7.5 on); row 24: d <= 1 (and, harmlessly, everything at or beyond the cut-off).
 */
#if defined(CPB_FINITE_LOG_ZERO) && !defined(CPB_LA_REPLICATED)
#define CPB_LA_COMPACT 1 /* default: the five-row table below; -DCPB_LA_REPLICATED builds the per-bucket, lane-replicated table */
#endif
#ifdef CPB_LA_COMPACT
/*
 * Compact table: five rows only -- the four segments and a row of zeros (the "polynomial" at and beyond the cut-off) -- in two
 * planes ({a,b} and {c,k}) of 128 bytes.  The rows of a plane lie in five different groups of four banks, so whatever rows the 32
 * lanes pick, a 128-bit fetch touches every bank with at most one address: one shared-memory wavefront per fetch (lanes that pick
 * the same row are served by broadcast), against four for a table with a row per lane.  The bucket -> row map is a 64-bit constant
 * of 2-bit fields, pre-shifted so that (MAP >> 2*bucket) & 0x30 is the row's byte offset.
 */
constexpr int LA_PLANE_DOUBLES = 16;                      /* 128 bytes: rows at 0, 16, 32, 48 (segments) and 64 (zeros) */
constexpr int LA_TABLE_DOUBLES = 2 * LA_PLANE_DOUBLES;
constexpr unsigned LA_ZERO_ROW = 64;
__host__ __device__ constexpr unsigned long long la_bucket_map() {
    unsigned long long m = 0;
    for (int r = 0; r < 24; r++) m |= (unsigned long long) (r <= 9 ? 1 : (r <= 16 ? 2 : 3)) << (2 * r + 4);
    return m;
}
__device__ __forceinline__ void fill_logadd_rows(double *la, int tid, int nthreads) {
    for (int i = tid; i < LA_TABLE_DOUBLES; i += nthreads) {
        const int plane = i / LA_PLANE_DOUBLES, row = (i % LA_PLANE_DOUBLES) / 2, e = i & 1;
        la[i] = row < 4 ? c_coefficients[4 * row + 2 * plane + e] : 0.0;
    }
}
typedef unsigned LaTable;
__device__ __forceinline__ LaTable logadd_lane_table(const double *la) { return (unsigned) __cvta_generic_to_shared(la); /* 128-byte aligned */ }
#else
#ifdef CPB_FINITE_LOG_ZERO
constexpr int LA_ROWS = 26; /* one more row of zeros: the "polynomial" at and beyond the cut-off */
#else
constexpr int LA_ROWS = 25;
#endif
/* Shared-memory layout of the table: two planes ({a,b} and {c,k}) of LA_ROWS rows; every row is replicated for the
 * 8 lanes of a quarter warp (8 x 16 bytes = all 32 banks), so a 128-bit fetch never has a bank conflict whatever
 * rows the lanes pick. */
constexpr int LA_ROW_DOUBLES = 16;                        /* 8 lanes x {2 doubles} */
constexpr int LA_PLANE_DOUBLES = LA_ROWS * LA_ROW_DOUBLES;
constexpr int LA_TABLE_DOUBLES = 2 * LA_PLANE_DOUBLES;    /* 6400 bytes */

__device__ __forceinline__ void fill_logadd_rows(double *la, int tid, int nthreads) {
    for (int i = tid; i < LA_TABLE_DOUBLES; i += nthreads) {
        const int plane = i / LA_PLANE_DOUBLES, r = (i % LA_PLANE_DOUBLES) / LA_ROW_DOUBLES, e = i & 1;
#ifdef CPB_FINITE_LOG_ZERO
        const int seg = r == 24 ? 0 : (r <= 9 ? 1 : (r <= 16 ? 2 : 3));
        la[i] = r == 25 ? 0.0 : c_coefficients[4 * seg + 2 * plane + e];
#else
        const int seg = r == LA_ROWS - 1 ? 0 : (r <= 9 ? 1 : (r <= 16 ? 2 : 3));
        la[i] = c_coefficients[4 * seg + 2 * plane + e];
#endif
    }
}
/* the calling lane's view of the table: the shared-memory byte address of its own 16-byte column */
typedef unsigned LaTable;
__device__ __forceinline__ LaTable logadd_lane_table(const double *la) {
    return (unsigned) __cvta_generic_to_shared(la) + 16u * (threadIdx.x & 7);
}
#endif

#ifdef CPB_LA_STATS
__device__ unsigned long long g_laStats[4]; /* warp-level calls, calls where every active lane is at or beyond the cut-off, lane calls, lane cut-offs */
#endif
#ifdef CPB_FINITE_LOG_ZERO
/*
 * Inside the kernels LOG_ZERO is the finite stand-in CPB_NEG_INF = -1e290 (see below): under this logAdd it behaves exactly as
 * -infinity does under the reference's (a term that far below the other operand is dropped, two of them give one of them back, sums
 * with finite terms stay "that far below"), and no infinity or NaN can reach the arithmetic.  That buys a cheaper operand selection:
 * beyond the cut-off the coefficient row is all zeros, so the polynomial is exactly 0 and the result is p + t with
 * t = the smaller operand (near) or the larger one (far) -- one 64-bit select instead of three.
 */
#ifdef CPB_LA_COMPACT
__device__ __forceinline__ double log_add(double x, double y, const LaTable la) {
    const double diff = __dsub_rn(x, y);
    const double d = fabs(diff);
    const bool far = !(d < 7.5);
    const bool pickX = (__double2hiint(diff) < 0) != far; /* near: x if it is the smaller; far: x if it is the larger */
    const int hi3 = __double2hiint(__dadd_rd(d, -4.9406564584124654e-324)); /* predecessor of d, see above */
    /* bucket = (hi3 >> 17) - 0x1FF8; below 0 (d <= 1) and from 24 on (beyond the cut-off anyway) the shift leaves no field: row 0 */
    int bucket; /* kept opaque so that the doubling below stays one multiply-add (FMA pipe) instead of a shift, a mask and an add (ALU pipe) */
    asm("shr.s32 %0, %1, 17;" : "=r"(bucket) : "r"(hi3));
    const unsigned sh = (unsigned) (bucket * 2 - 2 * 0x1FF8);
    unsigned long long f;
    asm("shr.u64 %0, %1, %2;" : "=l"(f) : "l"(la_bucket_map()), "r"(sh)); /* PTX clamps the shift amount at 64 */
    const unsigned row = far ? la + LA_ZERO_ROW : (((unsigned) f & 0x30u) | la);
    double a, b, c, k;
    asm("ld.shared.v2.f64 {%0, %1}, [%4];\n\tld.shared.v2.f64 {%2, %3}, [%4+%5];"
        : "=d"(a), "=d"(b), "=d"(c), "=d"(k)
        : "r"(row), "n"(LA_PLANE_DOUBLES * 8));
    double p = __dadd_rn(__dmul_rn(a, d), b);
    p = __dadd_rn(__dmul_rn(p, d), c);
    p = __dadd_rn(__dmul_rn(p, d), k);
    return __dadd_rn(p, pickX ? x : y);
}
#else
__device__ __forceinline__ double log_add(double x, double y, const LaTable la) {
    const double diff = __dsub_rn(x, y);
    const double d = fabs(diff);
    const bool far = !(d < 7.5);
    const bool pickX = (__double2hiint(diff) < 0) != far; /* near: x if it is the smaller; far: x if it is the larger */
    const int hi3 = __double2hiint(__dadd_rd(d, -4.9406564584124654e-324)); /* predecessor of d, see above */
    unsigned r = min((unsigned) ((hi3 >> 17) - 0x1FF8), 24u);
    r = far ? 25u : r;
    double a, b, c, k;
    asm("ld.shared.v2.f64 {%0, %1}, [%4];\n\tld.shared.v2.f64 {%2, %3}, [%4+%5];"
        : "=d"(a), "=d"(b), "=d"(c), "=d"(k)
        : "r"(la + (unsigned) (LA_ROW_DOUBLES * 8) * r), "n"(LA_PLANE_DOUBLES * 8));
    double p = __dadd_rn(__dmul_rn(a, d), b);
    p = __dadd_rn(__dmul_rn(p, d), c);
    p = __dadd_rn(__dmul_rn(p, d), k);
    return __dadd_rn(p, pickX ? x : y);
}
#endif
#else
__device__ __forceinline__ double log_add(double x, double y, const LaTable la) {
    const double diff = __dsub_rn(x, y);
#ifdef CPB_LA_STATS
    {
        const unsigned am = __activemask();
        const bool far = !(fabs(diff) < 7.5);
        const unsigned fm = __ballot_sync(am, far);
        if ((threadIdx.x & 31) == __ffs(am) - 1) {
            atomicAdd(&g_laStats[0], 1ull);
            if (fm == am) atomicAdd(&g_laStats[1], 1ull);
            atomicAdd(&g_laStats[2], (unsigned long long) __popc(am));
            atomicAdd(&g_laStats[3], (unsigned long long) __popc(fm));
        }
    }
#endif
    const bool xSmaller = __double2hiint(diff) < 0; /* sign of x-y; both -inf gives NaN, handled below */
    const double big = xSmaller ? y : x;
    const double small = xSmaller ? x : y;
    const double d = fabs(diff); /* a free operand modifier */
    /* bits(d) - 1 in one FP64 instruction: d minus the smallest denormal, rounded down, is the predecessor of d
     * (d = 0 gives a negative number, which like NaN and +inf ends up in the last row after the unsigned clamp) */
    const int hi3 = __double2hiint(__dadd_rd(d, -4.9406564584124654e-324));
    const unsigned r = min((unsigned) ((hi3 >> 17) - 0x1FF8), (unsigned) (LA_ROWS - 1));
    /* lanes at or beyond the cut-off all land in the last row, so they share one address per bank group */
    double a, b, c, k;
    asm("ld.shared.v2.f64 {%0, %1}, [%4];\n\tld.shared.v2.f64 {%2, %3}, [%4+%5];"
        : "=d"(a), "=d"(b), "=d"(c), "=d"(k)
        : "r"(la + (unsigned) (LA_ROW_DOUBLES * 8) * r), "n"(LA_PLANE_DOUBLES * 8));
    double p = __dadd_rn(__dmul_rn(a, d), b);
    p = __dadd_rn(__dmul_rn(p, d), c);
    p = __dadd_rn(__dmul_rn(p, d), k);
    p = __dadd_rn(p, small);
    /* d >= 7.5, d = +inf (one side is LOG_ZERO) and d = NaN (both are) all return the larger operand */
    return d < 7.5 ? p : big;
}
#endif

#define CPB_TRUE_NEG_INF (__longlong_as_double(0xFFF0000000000000LL))
#ifdef CPB_FINITE_LOG_ZERO
#define CPB_NEG_INF (-1e290)            /* LOG_ZERO inside the kernels: tables, initial states, band masks, planes */
#define CPB_IS_LOG_ZERO(v) (!((v) > -1e280)) /* anything that low is "log of zero" (sums of stand-ins included) */
#else
#define CPB_NEG_INF CPB_TRUE_NEG_INF
#define CPB_IS_LOG_ZERO(v) (false)
#endif

#ifndef CPB_STRIP_MIN_BLOCKS
#define CPB_STRIP_MIN_BLOCKS 4 /* resident CTAs per SM the wavefront kernels are compiled for (register budget) */
#endif
#ifndef CPB_FWD_MIN_BLOCKS
#define CPB_FWD_MIN_BLOCKS CPB_STRIP_MIN_BLOCKS
#endif
#ifndef CPB_BWD_MIN_BLOCKS
#define CPB_BWD_MIN_BLOCKS 6 /* backward gains 8 % from 24 resident warps per SM (80 registers); forward loses 5 %: it keeps 128 registers */
#endif
#ifndef CPB_BWD_WIDE_MIN_BLOCKS
#define CPB_BWD_WIDE_MIN_BLOCKS 3 /* very wide bands (engine.cu kBwdWideBand): 168 registers, no spills; 500 x 100 kb: 644 ms at 6 CTAs/SM, 582 at 5, 540 at 4, 504 at 3, 636 at 2 */
#endif

/* ---------------------------------------------------------------------------------------------
 * per-CTA tables: eP + tP for every (symbol, transition)
 * ------------------------------------------------------------------------------------------- */
template <int S> struct Shape;
template <> struct Shape<5> { static constexpr int NL = 4, NM = 5, NU = 4; };
template <> struct Shape<3> { static constexpr int NL = 3, NM = 3, NU = 3; };

template <int S> struct Tables {
    double tl[5][Shape<S>::NL];      /* [cX][k]  gap-X emission + lower transition */
    double tm[25][Shape<S>::NM];     /* [cX*5+cY][k] */
    double tu[5][Shape<S>::NU];      /* [cY][k] */
    double startv[S], rstartv[S], endv[S], rendv[S];
    double eGapX[5], eGapY[5], eMatch[25]; /* bare emissions: the DP kernels add the (uniform) transition per cell */
};

template <int S> __device__ __forceinline__ void fill_tables(Tables<S> &t, const CpbModel &m, int tid, int nthreads) {
    for (int i = tid; i < 5 * Shape<S>::NL; i += nthreads) {
        const int c = i / Shape<S>::NL, k = i % Shape<S>::NL;
        t.tl[c][k] = m.eGapX[c] + m.tLower[k];
    }
    for (int i = tid; i < 25 * Shape<S>::NM; i += nthreads) {
        const int c = i / Shape<S>::NM, k = i % Shape<S>::NM;
        t.tm[c][k] = m.eMatch[c] + m.tMiddle[k];
    }
    for (int i = tid; i < 5 * Shape<S>::NU; i += nthreads) {
        const int c = i / Shape<S>::NU, k = i % Shape<S>::NU;
        t.tu[c][k] = m.eGapY[c] + m.tUpper[k];
    }
    if (tid < 5) {
        t.eGapX[tid] = m.eGapX[tid];
        t.eGapY[tid] = m.eGapY[tid];
    }
    if (tid < 25) t.eMatch[tid] = m.eMatch[tid];
    if (tid < S) {
        t.startv[tid] = m.start[tid];
        t.rstartv[tid] = m.raggedStart[tid];
        t.endv[tid] = m.end[tid];
        t.rendv[tid] = m.raggedEnd[tid];
    }
}


/* (from, to) state of the k-th transition of each neighbour group, in the reference's issue order
 * (impl/stateMachine.c:454-479 five-state, :695-713 three-state) */
template <int S> __host__ __device__ constexpr int lower_from(int k) { return S == 5 ? (k == 0 ? 0 : (k == 1 ? 1 : (k == 2 ? 0 : 3))) : k; }
template <int S> __host__ __device__ constexpr int lower_to(int k) { return S == 5 ? (k < 2 ? 1 : 3) : 1; }
template <int S> __host__ __device__ constexpr int middle_from(int k) { return k; }
/* states that occur as the source of a lower / an upper transition (k_expect fetches only those) */
template <int S> __host__ __device__ constexpr bool uses_lower_from(int s) { return S == 5 ? (s == 0 || s == 1 || s == 3) : true; }
template <int S> __host__ __device__ constexpr bool uses_upper_from(int s) { return S == 5 ? (s == 0 || s == 2 || s == 4) : true; }
template <int S> __host__ __device__ constexpr int upper_from(int k) { return S == 5 ? (k == 0 ? 0 : (k == 1 ? 2 : (k == 2 ? 0 : 4))) : (k == 0 ? 0 : (k == 1 ? 2 : 1)); }
template <int S> __host__ __device__ constexpr int upper_to(int k) { return S == 5 ? (k < 2 ? 2 : 4) : 2; }

/* ---------------------------------------------------------------------------------------------
 * Two-pass forward (long regions): checkpoint bookkeeping.  A block's checkpoint is the full forward cells of its
 * diagonals T-1 and T, [state][cell], T-1 first.  The plane-less first pass writes them through the kernel's "aux"
 * stores: it runs on a copy of the diagonal records in which exactly the checkpoint diagonals carry an aux offset.
 * ------------------------------------------------------------------------------------------- */
__global__ void k_ckpt_sizes(const BlockRec *blocks, const RegionDev *regions, const DiagRec *diags, int nBlocks, int S, int32_t *sizes) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nBlocks) return;
    const BlockRec B = blocks[k];
    const DiagRec *dg = diags + regions[B.region].diagBase;
    sizes[k] = B.T > 0 ? S * (dg[B.T - 1].width + dg[B.T].width) : 0;
}
__global__ void k_ckpt_diags(const DiagRec *diags, DiagRec *out, int64_t n) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    DiagRec r = diags[i];
    r.aoff = NO_AUX;
    out[i] = r;
}
__global__ void k_ckpt_mark(const BlockRec *blocks, const RegionDev *regions, DiagRec *ckDiags, int nBlocks, int S) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nBlocks) return;
    const BlockRec B = blocks[k];
    if (B.T <= 0) return;
    DiagRec *dg = ckDiags + regions[B.region].diagBase;
    dg[B.T - 1].aoff = (uint32_t) B.ckBase;
    dg[B.T].aoff = (uint32_t) (B.ckBase + (int64_t) S * dg[B.T - 1].width);
}

/* ---------------------------------------------------------------------------------------------
 * k_totals : one warp per block, one lane per decade (10 owned diagonals share one totalProbability,
 * impl/pairwiseAligner.c:830-838).  Each fold is the reference's strictly sequential logAdd over the
 * cells of the diagonal (dpDiagonal_dotProduct, :513-523), so lanes run independent folds in parallel.
 * ------------------------------------------------------------------------------------------- */
__global__ void __launch_bounds__(128) k_totals(const DpArgs a, int nBlocks) {
    __shared__ __align__(128) double laTable[LA_TABLE_DOUBLES];
    fill_logadd_rows(laTable, threadIdx.x, blockDim.x);
    __syncthreads();
    const LaTable ctab = logadd_lane_table(laTable);
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= nBlocks) return;
    const BlockRec K = a.blocks[a.list[warp]];
    const RegionDev R = a.regions[K.region];
    const DiagRec *dg = a.diags + R.diagBase;
    const double *aux = a.aux + R.auxBase;
    const int nDecades = (K.from - K.T + 9) / 10;
    for (int j = lane; j < nDecades; j += 32) {
        const int dt = K.from - 10 * j;
        const DiagRec rec = dg[dt];
        const double *v = aux + rec.aoff + (int64_t) a.auxF * rec.width;
        double total = CPB_NEG_INF;
        for (int i = 0; i < rec.width; i++) total = log_add(total, v[i], ctab);
        if (dt + 1 <= K.top) {
            const int w2 = dg[dt + 1].width;
            const double *v2 = v + rec.width;
            double t2 = CPB_NEG_INF;
            for (int i = 0; i < w2; i++) t2 = log_add(t2, v2[i], ctab);
            total = log_add(total, t2, ctab);
        }
        a.totals[R.diagBase + dt] = total;
    }
}

/* ---------------------------------------------------------------------------------------------
 * k_posterior : one CTA of POST_WARPS warps per block, one warp per decade at a time.
 * The cells of a decade (10 owned diagonals sharing one totalProbability) are one contiguous range of the F+B
 * plane, so the scan is a flat, coalesced sweep:
 *   WRITE == false : evaluates exp(F+B-total) >= threshold for every cell (addPosteriorProb,
 *                    impl/pairwiseAligner.c:655-664), stores one ballot word per 32 cells and the number of kept
 *                    cells of the decade; cells on the matrix border (x = 0 / y = 0, which the reference skips,
 *                    :672, :700-729) are then struck out again -- at most two per diagonal;
 *   (device scan of the decade counts)
 *   WRITE == true  : revisits only the set bits, recovers (x, y) from the diagonal records and writes
 *                    (pInt, x, y) at the decade's offset.
 * Decades are numbered in ascending-diagonal order inside a block, so the output of a region is sorted by
 * (x+y, x).  Mask word of chunk-relative cell C in decade g: (C >> 5) + g -- the "+ g" keeps neighbouring
 * decades, whose cell ranges may share a 32-cell group, in different words.
 * ------------------------------------------------------------------------------------------- */
constexpr int POST_WARPS = 8;

/* A kept cell whose integer weight floor(p * 1e7) is not safe against the last-place difference between this device's exp and the
 * host's libm (the reference computes p with libm): the host recomputes it from the exact log-probability and patches the triple. */
struct PintFixup {
    double lp;    /* (F.M + B.M) - total, bit-identical to the reference's argument of exp */
    int64_t pos;  /* triple index in the output list */
    int32_t list; /* 0 match, 1 gap X, 2 gap Y */
    int32_t pad_;
};

struct PostArgs {
    double logThreshold;     /* smallest log-probability lp with exp(lp) >= threshold under the HOST's libm (host bisection, engine.cu):
                              * the keep decision is a comparison in log space, so it cannot differ from the reference's p >= threshold */
    double pintTolerance;    /* distance of p * 1e7 from an integer below which the host recomputes the weight (2e-8: three times the worst
                              * case of a 1-ulp device exp against a 1-ulp libm exp) */
    int32_t nLists;          /* 1 or 3 */
    int32_t fixupCap;
    int64_t nDecades;        /* decades in this chunk (stride between lists in counts/offsets) */
    int64_t maskWords;       /* mask words per list */
    int32_t *counts;         /* [nLists][nDecades] */
    const int64_t *offsets;  /* [nLists][nDecades] exclusive, global (WRITE) */
    uint32_t *masks;         /* [nLists][maskWords] */
    int32_t *out[3];
    unsigned int *fixupCount; /* WRITE: number of PintFixup records requested (may exceed fixupCap: the host then reports it) */
    PintFixup *fixups;
};

/* addPosteriorProb's test (impl/pairwiseAligner.c:656): p >= threshold, decided in log space (see PostArgs.logThreshold) */
__device__ __forceinline__ bool posterior_keep(double z, double total, const PostArgs &p) { return z - total >= p.logThreshold; }
/* addPosteriorProb's weight (:657-661): floor(min(p, 1) * 1e7); `safe` = the host's libm would give the same integer */
__device__ __forceinline__ int posterior_weight(double lp, const PostArgs &p, bool &safe) {
    double pr = exp(lp);
    if (pr > 1.0) pr = 1.0;
    const double v = pr * (double) CPB_PAIR_ALIGNMENT_PROB_1, fl = floor(v);
    /* lp >= 0 (F + B and the total agree to the last place, as they do for every confidently aligned cell: both are ~ -1e3 and their
     * difference is a multiple of 2e-13): exp gives >= 1 under any libm, the clamp makes it 1, the weight is 1e7 on both sides */
    /* (and below 1 - tolerance the weight is 0 on both sides however small p is: exp is never negative) */
    safe = lp >= 0.0 || ((fl == 0.0 || v - fl >= p.pintTolerance) && fl + 1.0 - v >= p.pintTolerance);
    return (int) fl;
}

template <bool WRITE>
__global__ void __launch_bounds__(32 * POST_WARPS) k_posterior(const DpArgs a, const PostArgs p) {
    __shared__ int sCoff[POST_WARPS][12], sXmyL[POST_WARPS][12]; /* WRITE: the current decade's diagonal records, per warp */
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const BlockRec K = a.blocks[a.list[blockIdx.x]];
    const RegionDev R = a.regions[K.region];
    const DiagRec *dg = a.diags + R.diagBase;
    const double *tot = a.totals + R.diagBase;
    const int nDecades = (K.from - K.T + 9) / 10;
    for (int j = warp; j < nDecades; j += POST_WARPS) {
        const int dt = K.from - 10 * j;                       /* the decade's total diagonal (its highest) */
        const int64_t g = K.decadeBase + (nDecades - 1 - j);  /* ascending-diagonal numbering */
        const double total = tot[dt];
        const bool alive = !CPB_IS_LOG_ZERO(total); /* no path through the decade: the reference's p is NaN there and nothing is kept */
        const int dLow = max(dt - 9, K.T + 1), nd = dt - dLow + 1;
        /* lane k < nd holds diagonal dLow + k */
        DiagRec mine;
        mine.xmyL = 0;
        mine.width = 0;
        mine.coff = 0;
        mine.aoff = 0;
        if (lane < nd) mine = dg[dLow + lane];
        const int64_t c0 = R.cellBase + __shfl_sync(0xFFFFFFFFu, mine.coff, 0);
        const int64_t c1 = R.cellBase + __shfl_sync(0xFFFFFFFFu, mine.coff, nd - 1) + __shfl_sync(0xFFFFFFFFu, mine.width, nd - 1);
        const int64_t cA = c0 & ~int64_t(31);
        for (int l = 0; l < p.nLists; l++) {
            const double *plane = a.planesB + (int64_t) l * a.planeStride;
            uint32_t *masks = p.masks + (int64_t) l * p.maskWords + g;
            if (!WRITE) {
                int cnt = 0;
                for (int64_t C = cA; C < c1; C += 128) {
                    double z[4];
                    bool valid[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int64_t cell = C + 32 * u + lane;
                        valid[u] = cell >= c0 && cell < c1;
                        z[u] = valid[u] ? __ldcs(plane + cell) : CPB_NEG_INF;
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const unsigned m = __ballot_sync(0xFFFFFFFFu, valid[u] && alive && posterior_keep(z[u], total, p));
                        if (C + 32 * u < c1) {
                            if (lane == 0) masks[(C >> 5) + u] = m;
                            cnt += __popc(m);
                        }
                    }
                }
                __syncwarp();
                /* strike out the border cells: list 0 (match) needs x > 0 and y > 0, list 1 (gap X) x > 0, list 2 (gap Y) y > 0 */
                int struck = 0;
                if (lane < nd) {
                    const int d = dLow + lane, xlo = (d + mine.xmyL) >> 1;
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        /* e = 0: the cell with x = 0 (first cell, if the diagonal starts in row 0); e = 1: the cell with y = 0 (x = d) */
                        const int i = e == 0 ? 0 : d - xlo;
                        const bool exists = e == 0 ? xlo == 0 : (i >= 0 && i < mine.width);
                        const bool applies = l == 0 || (l == 1 && e == 0) || (l == 2 && e == 1);
                        if (exists && applies) {
                            const int64_t cell = R.cellBase + mine.coff + i;
                            const uint32_t bit = 1u << (cell & 31);
                            if (atomicAnd(masks + (cell >> 5), ~bit) & bit) struck++; /* (0,0) may be visited twice: the second visit finds the bit gone */
                        }
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) struck += __shfl_xor_sync(0xFFFFFFFFu, struck, o);
                if (lane == 0) p.counts[(int64_t) l * p.nDecades + g] = cnt - struck;
            } else {
                /* Kept cells are rare (about one per diagonal).  32 mask words of the decade at a time: every lane takes one word, a warp
                 * scan numbers the set bits of the group, and then every lane takes one KEPT CELL -- it finds the word that holds its
                 * cell by bisection over the scan and the bit inside it with __fns.  (A lane per word, each writing out its own word's
                 * bits, left 28 lanes idle on narrow bands, where a decade is three or four words: 20 of 145 ms per 100 000 x 1 kb
                 * pairs with cPecanRealign's band.)  The decade's records sit in shared memory for the per-lane diagonal search. */
                int64_t run = p.offsets[(int64_t) l * p.nDecades + g];
                __syncwarp();
                if (lane < nd) {
                    sCoff[warp][lane] = (int) mine.coff;
                    sXmyL[warp][lane] = mine.xmyL;
                }
                __syncwarp();
                const int64_t nWords = (c1 - cA + 31) >> 5;
                for (int64_t wb = 0; wb < nWords; wb += 32) {
                    const int64_t wi = wb + lane;
                    const unsigned m = wi < nWords ? masks[(cA >> 5) + wi] : 0u;
                    const int cnt = __popc(m);
                    int incl = cnt;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                        if (lane >= o) incl += t;
                    }
                    const int kept = __shfl_sync(0xFFFFFFFFu, incl, 31);
                    for (int t0 = 0; t0 < kept; t0 += 32) {
                        const int t = t0 + lane; /* this lane's kept cell of the group, if t < kept */
                        /* the first word whose inclusive count exceeds t */
                        int w = 0;
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            const int probe = __shfl_sync(0xFFFFFFFFu, incl, w + o - 1);
                            if (probe <= t) w += o;
                        }
                        w = min(w, 31);
                        const unsigned mw = __shfl_sync(0xFFFFFFFFu, m, w);
                        const int before = __shfl_sync(0xFFFFFFFFu, incl, w) - __popc(mw);
                        if (t < kept) {
                            const int bit = (int) __fns(mw, 0, t - before + 1);
                            const int64_t cell = cA + ((wb + w) << 5) + bit;
                            /* the diagonal of the cell: the last of the decade's diagonals that starts at or before it */
                            int k = 0;
                            for (int q = 1; q < nd; q++) k = cell >= R.cellBase + sCoff[warp][q] ? q : k;
                            const int d = dLow + k;
                            const int x = ((d + sXmyL[warp][k]) >> 1) + (int) (cell - R.cellBase - sCoff[warp][k]), y = d - x;
                            const int64_t pos = run + t;
                            bool safe;
                            const double lp = plane[cell] - total;
                            const int pInt = posterior_weight(lp, p, safe);
                            if (!safe) {
                                const unsigned k = atomicAdd(p.fixupCount, 1u);
                                if (k < (unsigned) p.fixupCap) {
                                    PintFixup f;
                                    f.lp = lp;
                                    f.pos = pos;
                                    f.list = l;
                                    f.pad_ = 0;
                                    p.fixups[k] = f;
                                }
                            }
                            int32_t *o = p.out[l] + 3 * pos;
                            o[0] = pInt;
                            o[1] = x - 1 + R.ox;
                            o[2] = y - 1 + R.oy;
                        }
                    }
                    run += kept;
                }
            }
        }
    }
}

/* ---- exclusive scan of int32 counts into int64 offsets (three small kernels) ---- */
constexpr int SCAN_TILE = 2048;

__global__ void __launch_bounds__(256) k_scan_tiles(const int32_t *counts, int64_t n, int64_t *tileSums) {
    __shared__ int64_t red[256];
    const int64_t base = (int64_t) blockIdx.x * SCAN_TILE;
    int64_t s = 0;
    for (int k = threadIdx.x; k < SCAN_TILE; k += 256) {
        const int64_t i = base + k;
        if (i < n) s += counts[i];
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) tileSums[blockIdx.x] = red[0];
}

/* single thread block: exclusive scan of the tile sums, starting from *startAt; writes the grand total to *totalOut */
__global__ void __launch_bounds__(1) k_scan_sums(int64_t *tileSums, int64_t nTiles, int64_t startAt, int64_t *totalOut) {
    int64_t run = startAt;
    for (int64_t t = 0; t < nTiles; t++) {
        const int64_t v = tileSums[t];
        tileSums[t] = run;
        run += v;
    }
    *totalOut = run;
}

__global__ void __launch_bounds__(256) k_scan_apply(const int32_t *counts, int64_t n, const int64_t *tileOff, int64_t *offsets) {
    /* each thread owns 8 consecutive elements of the tile */
    __shared__ int64_t part[256];
    const int64_t base = (int64_t) blockIdx.x * SCAN_TILE + (int64_t) threadIdx.x * 8;
    int32_t v[8];
    int64_t s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        v[k] = base + k < n ? counts[base + k] : 0;
        s += v[k];
    }
    part[threadIdx.x] = s;
    __syncthreads();
    /* Hillis-Steele inclusive scan over 256 partials */
    for (int o = 1; o < 256; o <<= 1) {
        int64_t t = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
        __syncthreads();
        part[threadIdx.x] += t;
        __syncthreads();
    }
    int64_t run = tileOff[blockIdx.x] + part[threadIdx.x] - s;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        if (base + k < n) offsets[base + k] = run;
        run += v[k];
    }
}

/* per pair: add the kept-cell counts of its decades in this chunk; decades of a pair are contiguous */
__global__ void k_pair_counts(const int32_t *counts, int64_t nDecades, int nLists, const int64_t *pairDecade0, int nPairs, int64_t *pairCounts,
                              int64_t pairStride) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nPairs * nLists) return;
    const int l = i / nPairs, q = i % nPairs;
    int64_t s = 0;
    for (int64_t g = pairDecade0[q]; g < pairDecade0[q + 1]; g++) s += counts[(int64_t) l * nDecades + g];
    pairCounts[(int64_t) l * pairStride + q] += s;
}

/* ---------------------------------------------------------------------------------------------
 * Post-posterior filters on the compacted output (SURVEY.md section 8f, N2): the AMAP-style gap reweighting
 * (getIndelProbabilities / reweightAlignedPairs, impl/pairwiseAligner.c:1519-1560) and the per-pair alignment score
 * (getAlignmentScore, impl/multipleAligner.c:604-619).  Integer sums, so atomics give the reference's result whatever the order.
 * ------------------------------------------------------------------------------------------- */
__device__ __forceinline__ int pair_of_triple(const int64_t *pairOff, int nPairs, int64_t t) {
    int lo = 0, hi = nPairs; /* last pair with pairOff[pair] <= t */
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (pairOff[mid] <= t) lo = mid;
        else hi = mid;
    }
    return lo;
}
__global__ void k_fill_i64(long long *p, int64_t n, long long v) {
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) p[i] = v;
}
/* gapX[xOff[pair] + x] and gapY[yOff[pair] + y] start at PAIR_ALIGNMENT_PROB_1; every aligned pair takes its weight off both */
__global__ void k_gap_weights(const int32_t *triples, int64_t nTriples, const int64_t *pairOff, int nPairs, const int64_t *xOff, const int64_t *yOff,
                              long long *gapX, long long *gapY) {
    const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nTriples) return;
    const int pair = pair_of_triple(pairOff, nPairs, t);
    const long long w = triples[3 * t];
    atomicAdd(reinterpret_cast<unsigned long long *>(gapX + xOff[pair] + triples[3 * t + 1]), (unsigned long long) (-w));
    atomicAdd(reinterpret_cast<unsigned long long *>(gapY + yOff[pair] + triples[3 * t + 2]), (unsigned long long) (-w));
}
/* weight - gapGamma * (gap weight of x + gap weight of y), gap weights floored at 0, the result truncated towards zero (:1536-1547) */
__global__ void k_reweight(int32_t *triples, int64_t nTriples, const int64_t *pairOff, int nPairs, const int64_t *xOff, const int64_t *yOff,
                           const long long *gapX, const long long *gapY, double gapGamma) {
    const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nTriples) return;
    const int pair = pair_of_triple(pairOff, nPairs, t);
    const long long gx = max(gapX[xOff[pair] + triples[3 * t + 1]], 0ll), gy = max(gapY[yOff[pair] + triples[3 * t + 2]], 0ll);
    triples[3 * t] = (int32_t) (long long) ((double) triples[3 * t] - gapGamma * (double) (gx + gy));
}
/* one warp per pair: the sum of its weights, normalised by the shorter sequence, clamped to [0, 1], in units of 1e-7 */
__global__ void k_alignment_scores(const int32_t *triples, const int64_t *pairOff, int nPairs, const int64_t *xOff, const int64_t *yOff, int64_t *scores) {
    const int pair = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (pair >= nPairs) return;
    long long sum = 0;
    for (int64_t t = pairOff[pair] + lane; t < pairOff[pair + 1]; t += 32) sum += triples[3 * t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xFFFFFFFFu, sum, o);
    if (lane == 0) {
        const int64_t l1 = xOff[pair + 1] - xOff[pair], l2 = yOff[pair + 1] - yOff[pair];
        int64_t j = l1 < l2 ? l1 : l2;
        j = j == 0 ? 1 : j;
        double d = (double) sum / (double) (j * (int64_t) CPB_PAIR_ALIGNMENT_PROB_1);
        d = d > 1.0 ? 1.0 : d;
        d = d < 0.0 ? 0.0 : d;
        scores[pair] = (int64_t) (d * CPB_PAIR_ALIGNMENT_PROB_1);
    }
}

/* ---------------------------------------------------------------------------------------------
 * k_expect : one warp per block; expected transition and emission counts
 * (diagonalCalculationExpectations / updateExpectations, impl/pairwiseAligner.c:418-438, :735-746)
 * partial[block][CPB_HMM_LEN(S)]
 * ------------------------------------------------------------------------------------------- */
constexpr int EXPECT_SHARE = 4, EXPECT_COLS = 32 / EXPECT_SHARE;
template <int S>
__global__ void __launch_bounds__(32, S == 5 ? 20 : 16) k_expect(const DpArgs a, const CpbModel model, double *partials) {
    extern __shared__ __align__(16) unsigned char smemRaw[];
    Tables<S> &tab = *reinterpret_cast<Tables<S> *>(smemRaw);
    /* emission accumulators [S*16][EXPECT_COLS]: a column is shared by EXPECT_SHARE neighbouring lanes, which add to it one after
     * the other (fixed order, so the sums are reproducible); 5 KB instead of 20 KB per warp lets four times as many warps stay
     * resident, and this kernel is a chain of dependent loads and exponentials that needs them */
    double *ePriv = reinterpret_cast<double *>(smemRaw + ((sizeof(Tables<S>) + 15) & ~size_t(15)));
    const int lane = threadIdx.x;
    const BlockRec K = a.blocks[a.list[blockIdx.x]];
    const RegionDev R = a.regions[K.region];
    fill_tables<S>(tab, model, lane, 32);
    for (int i = lane; i < S * 16 * EXPECT_COLS; i += 32) ePriv[i] = 0.0;
    __syncwarp();
    const DiagRec *dg = a.diags + R.diagBase;
    const uint8_t *sx = a.symX + R.xBase, *sy = a.symY + R.yBase;
    const double *pf = a.planesF + R.cellBase, *pb = a.planesB + R.cellBase;
    const double *tot = a.totals + R.diagBase;
    constexpr int NL = Shape<S>::NL, NM = Shape<S>::NM, NU = Shape<S>::NU;
    double accT[NL + NM + NU];
#pragma unroll
    for (int k = 0; k < NL + NM + NU; k++) accT[k] = 0.0;
    double likelihood = 0.0;

    /* The owned cells of a decade (10 diagonals sharing one totalProbability) are one contiguous range of the cell enumeration:
     * lanes sweep it flat, 32 cells at a time whatever the band width, and find their diagonal among the decade's records, which
     * lanes 0..nd+1 hold (two more below the decade for the lower / upper and middle neighbours). */
    const int nDecades = (K.from - K.T + 9) / 10;
    for (int j = 0; j < nDecades; j++) {
        const int dt = K.from - 10 * j, dLow = max(dt - 9, K.T + 1), nd = dt - dLow + 1;
        const double total = tot[dt];
        for (int q = 0; q < nd; q++) likelihood += CPB_IS_LOG_ZERO(total) ? CPB_TRUE_NEG_INF : total; /* once per diagonal (impl/pairwiseAligner.c:743), highest first */
        /* No path through the decade (the band forces a transition the model forbids): the reference computes exp(-inf - -inf) = NaN for
         * every term it adds there, and so do we */
        const double minusTotal = CPB_IS_LOG_ZERO(total) ? __longlong_as_double(0x7FF8000000000000LL) : -total;
        DiagRec mine = dg[max(dLow - 2 + min(lane, nd + 1), 0)]; /* lane r: diagonal dLow - 2 + r */
        const int c0 = (int) __shfl_sync(0xFFFFFFFFu, mine.coff, 2);
        const int c1 = (int) (__shfl_sync(0xFFFFFFFFu, mine.coff, nd + 1) + __shfl_sync(0xFFFFFFFFu, (uint32_t) mine.width, nd + 1));
        /* first cell of the decade's 2nd .. 10th diagonal (beyond nd: never reached), fetched once per decade, not once per 32 cells */
        int firstCell[9];
#pragma unroll
        for (int t = 1; t < 10; t++) {
            const int ct = (int) __shfl_sync(0xFFFFFFFFu, mine.coff, min(t, nd - 1) + 2);
            firstCell[t - 1] = t < nd ? ct : 0x7FFFFFFF;
        }
        for (int base = c0; base < c1; base += 32) {
            const int c = base + lane;
            const bool valid = c < c1;
            int q = 0;
#pragma unroll
            for (int t = 1; t < 10; t++) q = c >= firstCell[t - 1] ? t : q;
            DiagRec rec, rec1, rec2;
            rec.xmyL = __shfl_sync(0xFFFFFFFFu, mine.xmyL, q + 2);
            rec.width = __shfl_sync(0xFFFFFFFFu, mine.width, q + 2);
            rec.coff = __shfl_sync(0xFFFFFFFFu, mine.coff, q + 2);
            rec1.xmyL = __shfl_sync(0xFFFFFFFFu, mine.xmyL, q + 1);
            rec1.width = __shfl_sync(0xFFFFFFFFu, mine.width, q + 1);
            rec1.coff = __shfl_sync(0xFFFFFFFFu, mine.coff, q + 1);
            rec2.xmyL = __shfl_sync(0xFFFFFFFFu, mine.xmyL, q);
            rec2.width = __shfl_sync(0xFFFFFFFFu, mine.width, q);
            rec2.coff = __shfl_sync(0xFFFFFFFFu, mine.coff, q);
            double q2[S]; /* per to-state sum for the emission expectation */
#pragma unroll
            for (int s = 0; s < S; s++) q2[s] = 0.0;
            bool emit = false;
            int eIdx = 0;
            if (valid) {
            const int d = dLow + q;
            const int i = c - (int) rec.coff;
            const bool haveM = d >= 2 && !(K.T > 0 && d == K.T + 1); /* F[d-2] was freed at the block boundary (:855) */
            const int xmy = rec.xmyL + 2 * i;
            const int x = (d + xmy) >> 1, y = (d - xmy) >> 1;
            const int iL = (xmy - 1 - rec1.xmyL) >> 1, iU = iL + 1; /* xmy-1 and xmy+1 on d-1 (same parity as rec1.xmyL) */
            const bool inL = xmy - 1 >= rec1.xmyL && iL < rec1.width;
            const bool inU = xmy + 1 >= rec1.xmyL && iU < rec1.width;
            const int iM = (xmy - rec2.xmyL) >> 1;
            const bool inM = haveM && xmy >= rec2.xmyL && iM < rec2.width;
            /* Every load of the cell is issued before the first exponential: the B states of the cell and the F states of its three
             * neighbours (a neighbour outside the band reads the cell itself -- a valid address whose value is not used).  Issued
             * inside the three branches below, the loads of one neighbour waited for the exponentials of the one before; the kernel
             * is bound by the latency of these loads (ncu: long scoreboard 4.2 stalled warps per issue). */
            const int64_t cell = c;
            const int64_t cellL = inL ? (int64_t) rec1.coff + iL : cell, cellU = inU ? (int64_t) rec1.coff + iU : cell, cellM = inM ? (int64_t) rec2.coff + iM : cell;
            const int cX = x > 0 ? sx[x - 1] : 4, cY = y > 0 ? sy[y - 1] : 4;
            double b[S], fL[S], fM[S], fU[S];
#pragma unroll
            for (int s = 0; s < S; s++) b[s] = pb[(int64_t) s * a.planeStride + cell];
#pragma unroll
            for (int s = 0; s < S; s++) {
                fM[s] = pf[(int64_t) s * a.planeStride + cellM];
                if (uses_lower_from<S>(s)) fL[s] = pf[(int64_t) s * a.planeStride + cellL];
                if (uses_upper_from<S>(s)) fU[s] = pf[(int64_t) s * a.planeStride + cellU];
            }
            emit = cX < 4 && cY < 4;
            eIdx = cX * 4 + cY;
            if (inL) {
#pragma unroll
                for (int k = 0; k < NL; k++) {
                    const int f = lower_from<S>(k), t = lower_to<S>(k);
                    const double pr = exp(fL[f] + b[t] + tab.tl[cX][k] + minusTotal);
                    accT[k] += pr;
                    q2[t] += pr;
                }
            }
            if (inM) {
#pragma unroll
                for (int k = 0; k < NM; k++) {
                    const int f = middle_from<S>(k);
                    const double pr = exp(fM[f] + b[0] + tab.tm[cX * 5 + cY][k] + minusTotal);
                    accT[NL + k] += pr;
                    q2[0] += pr;
                }
            }
            if (inU) {
#pragma unroll
                for (int k = 0; k < NU; k++) {
                    const int f = upper_from<S>(k), t = upper_to<S>(k);
                    const double pr = exp(fU[f] + b[t] + tab.tu[cY][k] + minusTotal);
                    accT[NL + NM + k] += pr;
                    q2[t] += pr;
                }
            }
            }
            for (int ph = 0; ph < EXPECT_SHARE; ph++) {
                if ((lane & (EXPECT_SHARE - 1)) == ph && emit) {
#pragma unroll
                    for (int s = 0; s < S; s++) ePriv[(s * 16 + eIdx) * EXPECT_COLS + lane / EXPECT_SHARE] += q2[s];
                }
                __syncwarp();
            }
        }
    }
    /* reduce over lanes in a fixed order and write this block's partial Hmm */
    double *out = partials + (int64_t) blockIdx.x * CPB_HMM_LEN(S);
    auto reduce = [&](double v) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
        return v;
    };
    double tsum[NL + NM + NU];
#pragma unroll
    for (int k = 0; k < NL + NM + NU; k++) tsum[k] = reduce(accT[k]);
    if (lane == 0) {
        for (int i = 0; i < S * S; i++) out[i] = 0.0;
#pragma unroll
        for (int k = 0; k < NL; k++) out[lower_from<S>(k) * S + lower_to<S>(k)] += tsum[k];
#pragma unroll
        for (int k = 0; k < NM; k++) out[middle_from<S>(k) * S + 0] += tsum[NL + k];
#pragma unroll
        for (int k = 0; k < NU; k++) out[upper_from<S>(k) * S + upper_to<S>(k)] += tsum[NL + NM + k];
        out[S * S + S * 16] = likelihood;
    }
    for (int i = 0; i < S * 16; i++) {
        const double v = reduce(lane < EXPECT_COLS ? ePriv[i * EXPECT_COLS + lane] : 0.0);
        if (lane == 0) out[S * S + i] = v;
    }
}

/* sum block partials per pair (blocks of a pair are contiguous and in order), one thread per (pair, entry) */
__global__ void k_reduce_pairs(const double *partials, const int64_t *pairBlockOff, int nPairs, int len, double *perPair) {
    const int64_t idx = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t) nPairs * len) return;
    const int pair = (int) (idx / len), e = (int) (idx % len);
    double s = 0.0;
    for (int64_t b = pairBlockOff[pair]; b < pairBlockOff[pair + 1]; b++) s += partials[b * len + e];
    perPair[idx] += s;
}

/* total over pairs: one CTA per entry (len <= 106); thread t adds pairs t, t + 256, ... in order, then a fixed tree over the 256
 * partial sums => the same bits on every run of the same batch (a single sequential chain of 50 000 adds took 4.6 ms) */
__global__ void __launch_bounds__(256) k_reduce_total(const double *perPair, int nPairs, int len, double *total) {
    __shared__ double part[256];
    const int e = blockIdx.x;
    double s = 0.0;
    for (int p = threadIdx.x; p < nPairs; p += 256) s += perPair[(int64_t) p * len + e];
    part[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int) threadIdx.x < o) part[threadIdx.x] += part[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) total[e] = part[0];
}

/* ---------------------------------------------------------------------------------------------
 * k_encode : chars -> symbols a,c,g,t,n = 0..4 (symbol_convertCharToSymbol, impl/pairwiseAligner.c:317-334), in place; the bytes
 * themselves, upper-cased as C's toupper does (only a-z change), go to `kept` for the decoders (left shift and identity compare bytes)
 * ------------------------------------------------------------------------------------------- */
__global__ void k_encode(uint8_t *s, uint8_t *kept, int64_t n) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t raw = s[i];
    kept[i] = raw >= 'a' && raw <= 'z' ? (uint8_t) (raw - ('a' - 'A')) : raw;
    const uint8_t c = raw & 0xDF; /* fold case */
    s[i] = c == 'A' ? 0 : (c == 'C' ? 1 : (c == 'G' ? 2 : (c == 'T' ? 3 : 4)));
}

/* ---------------------------------------------------------------------------------------------
 * k_split_flags : one warp per pair -- where getSplitPoints (impl/pairwiseAligner.c:1230-1257) cuts a pair into regions.
 * Pair i has nA + 1 gaps: gap g lies between anchor g-1 (or the origin) and anchor g (or the end of both sequences).  Bit
 * aOff[i] + i + g of `flags` is set iff the rectangle of gap g holds more than splitBiggerThan cells.  The host turns the flagged
 * gaps into region records without walking the anchors itself (the anchors of 100 000 x 1 kb pairs are a gigabyte).
 * ------------------------------------------------------------------------------------------- */
__global__ void k_split_flags(const int32_t *anchors, const int64_t *aOff, const int64_t *xOff, const int64_t *yOff, int nPairs, long long splitBiggerThan,
                              uint32_t *flags, unsigned int *nFlaggedPairs) {
    const int pair = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pair >= nPairs) return;
    const int64_t a0 = aOff[pair], nA = aOff[pair + 1] - a0;
    const int64_t lX = xOff[pair + 1] - xOff[pair], lY = yOff[pair + 1] - yOff[pair];
    const int32_t *an = anchors + 3 * a0;
    const int64_t bit0 = a0 + pair;
    bool any = false;
    for (int64_t g0 = 0; g0 <= nA; g0 += 32) {
        const int64_t g = g0 + lane;
        bool f = false;
        if (g <= nA) {
            const int64_t prevX = g > 0 ? (int64_t) an[3 * (g - 1)] + 1 : 0, prevY = g > 0 ? (int64_t) an[3 * (g - 1) + 1] + 1 : 0;
            const int64_t nextX = g < nA ? (int64_t) an[3 * g] : lX, nextY = g < nA ? (int64_t) an[3 * g + 1] : lY;
            f = (nextX - prevX) * (nextY - prevY) > splitBiggerThan;
        }
        const unsigned m = __ballot_sync(0xFFFFFFFFu, f);
        if (m != 0 && lane == 0) {
            const int64_t B = bit0 + g0;
            const int sh = (int) (B & 31);
            atomicOr(flags + (B >> 5), m << sh);
            if (sh != 0 && (m >> (32 - sh)) != 0) atomicOr(flags + (B >> 5) + 1, m >> (32 - sh));
            any = true;
        }
    }
    if (lane == 0 && any) atomicAdd(nFlaggedPairs, 1u);
}

/* ---------------------------------------------------------------------------------------------
 * k_band : one warp per region -- the device-side band builder and traceback scheduler.
 *   band:     band_construct / band_constructDynamic, impl/pairwiseAligner.c:94-234.  The reference walks the diagonals
 *             with a moving (previous anchor, next anchor) pair; here every lane takes one diagonal, finds its anchor
 *             interval by binary search (anchors are strictly increasing in x+y) and evaluates the same box formula.
 *   schedule: the traceback trigger of getPosteriorProbsWithBanding, :791-793, :810, :830, :852, found with ballots.
 * ------------------------------------------------------------------------------------------- */
struct BandArgs {
    RegionDev *regions;
    const int32_t *anchors; /* (x,y,expansion) triples, pair coordinates */
    DiagRec *diags;
    BlockRec *blocks;
    StripRec *strips;
    int32_t nRegions;
    int32_t expansion, dynamic;
    int32_t minDiags, traceBack;
    int32_t auxF;       /* full-F planes in the aux record of a total diagonal */
    int32_t scheduleOn; /* 0: forward-only, no blocks */
};

__device__ __forceinline__ int64_t clamp_coord(int64_t z, int64_t l) { return z < 0 ? 0 : (z > l ? l : z); }

constexpr int BAND_WARPS = 4;

__global__ void __launch_bounds__(32 * BAND_WARPS) k_band(const BandArgs b) {
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * BAND_WARPS + (threadIdx.x >> 5);
    if (r >= b.nRegions) return;
    const unsigned FULL = 0xFFFFFFFFu;
    RegionDev R = b.regions[r];
    DiagRec *dg = b.diags + R.diagBase;
    const int32_t *an = b.anchors + 3 * R.anchorBase;
    const int nA = R.nAnchors;
    const int64_t lX = R.lX, lY = R.lY, N = lX + lY;
    StripRec *st = b.strips + R.stripBase;
    const int nStrips = (int) (lX >> 5) + 1;
    for (int k = lane; k < nStrips; k += 32) {
        st[k].dFirst = 0x7FFFFFFF;
        st[k].dLast = -1;
    }
    __syncwarp();
    /* anchor i in matrix coordinates of the region */
    auto axay = [&](int i) { return (int64_t) an[3 * i] - R.ox + 1 + (int64_t) an[3 * i + 1] - R.oy + 1; };

    int err = 0, maxW = 0;
    int64_t cellsBefore = 0;       /* cells of all diagonals before this chunk */
    int aLo = 0;                   /* first anchor whose x+y is >= the chunk's first diagonal */
    int carryLo = 0, carryHi = -1; /* strips touched by the last diagonal of the previous chunk */
    for (int64_t base = 0; base <= N; base += 32) {
        const int64_t xay = base + lane;
        const bool live = xay <= N;
        int64_t l = 0, rr = 0;
        int n = aLo;
        if (live && xay > 0) {
            /* n = first anchor with x+y >= xay: at most 16 anchors (x+y grows by >= 2) lie inside the chunk */
            int lo = aLo, hi = min(nA, aLo + 17);
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (axay(mid) < xay) lo = mid + 1;
                else hi = mid;
            }
            n = lo;
            int64_t px = 0, py = 0, nx = lX, ny = lY, e = b.dynamic ? 0 : b.expansion;
            if (n > 0) {
                px = (int64_t) an[3 * (n - 1)] - R.ox + 1;
                py = (int64_t) an[3 * (n - 1) + 1] - R.oy + 1;
            }
            if (n < nA) {
                nx = (int64_t) an[3 * n] - R.ox + 1;
                ny = (int64_t) an[3 * n + 1] - R.oy + 1;
                if (b.dynamic) e = an[3 * n + 2];
            } else if (b.dynamic && nA > 0) {
                e = an[3 * (nA - 1) + 2]; /* past the last anchor the reference keeps that anchor's expansion */
            }
            const int64_t pxay = px + py, pxmy = px - py, nxay = nx + ny, nxmy = nx - ny;
            const int64_t xL = clamp_coord((pxay + (pxmy - e)) / 2, lX), yL = clamp_coord((nxay - (nxmy - e)) / 2, lY);
            const int64_t xU = clamp_coord((nxay + (nxmy + e)) / 2, lX), yU = clamp_coord((pxay - (pxmy + e)) / 2, lY);
            int64_t v;
            l = xL - yL;
            rr = xU - yU;
            if ((xay + l) % 2 != 0) l += 1;
            if ((xay + rr) % 2 != 0) rr += 1;
            v = (xay + l) / 2; if (v < xL) l += 2 * (xL - v);
            v = (xay - l) / 2; if (yL < v) l += 2 * (v - yL);
            v = (xay + rr) / 2; if (xU < v) rr -= 2 * (v - xU);
            v = (xay - rr) / 2; if (v < yU) rr -= 2 * (yU - v);
            if ((xay + l) % 2 != 0 || (xay + rr) % 2 != 0 || l > rr) {
                err = 1;
                rr = l; /* keep the tables well-formed; the host reports the error */
            }
        }
        const int w = live ? (int) ((rr - l) / 2 + 1) : 0;
        /* cell offsets: exclusive prefix sum of the widths */
        int incl = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += t;
        }
        if (live) {
            DiagRec rec;
            rec.xmyL = (int32_t) l;
            rec.width = w;
            rec.coff = (uint32_t) (cellsBefore + incl - w);
            rec.aoff = NO_AUX;
            dg[xay] = rec;
        }
        cellsBefore += __shfl_sync(FULL, incl, 31);
        maxW = max(maxW, w);
        /* 32-row strips touched by this diagonal: rows (xay + l)/2 .. (xay + rr)/2; record where strips enter and leave */
        int sLo = live ? (int) (((xay + l) / 2) >> 5) : 0, sHi = live ? min((int) (((xay + rr) / 2) >> 5), nStrips - 1) : -1;
        int pLo = __shfl_up_sync(FULL, sLo, 1), pHi = __shfl_up_sync(FULL, sHi, 1);
        if (lane == 0) {
            pLo = carryLo;
            pHi = carryHi;
        }
        if (live) {
            for (int k = sLo; k <= sHi; k++) {
                if (k < pLo || k > pHi) atomicMin(&st[k].dFirst, (int) xay);
            }
            for (int k = pLo; k <= pHi; k++) {
                if (k < sLo || k > sHi) atomicMax(&st[k].dLast, (int) xay - 1);
            }
        }
        /* carry the state of the chunk's last live diagonal */
        const int lastLive = N - base < 31 ? (int) (N - base) : 31;
        carryLo = __shfl_sync(FULL, sLo, lastLive);
        carryHi = __shfl_sync(FULL, sHi, lastLive);
        aLo = __shfl_sync(FULL, n, lastLive);
        /* the next chunk starts one diagonal later: its first anchor is the first with x+y >= base+32, i.e. n of the last lane, unless that anchor lies exactly on it */
        if (aLo < nA && axay(aLo) < base + 32) aLo++;
    }
    for (int k = carryLo + lane; k <= carryHi; k += 32) atomicMax(&st[k].dLast, (int) N); /* strips still touched by the last diagonal */
    if (lane == 0) {
        DiagRec sentinel;
        sentinel.xmyL = 0;
        sentinel.width = 0;
        sentinel.coff = (uint32_t) cellsBefore;
        sentinel.aoff = NO_AUX;
        dg[N + 1] = sentinel;
        dg[N + 2] = sentinel;
    }
    __syncwarp();

    /* ---- traceback schedule ---- */
    int nBlocks = 0;
    int64_t auxD = 0;
    if (b.scheduleOn && N > 0) {
        BlockRec *bl = b.blocks + R.blockBase;
        const int thresholdW = 2 * b.expansion + 1;
        int64_t T = 0;
        for (;;) {
            /* the next traceback point: the first diagonal >= T + minDiags that is narrow enough, or N */
            int64_t d = N;
            for (int64_t q = T + b.minDiags; q < N; q += 32) {
                const int64_t k = q + lane;
                const bool hit = k < N && dg[k].width <= thresholdW;
                const unsigned m = __ballot_sync(FULL, hit);
                if (m != 0) {
                    d = q + __ffs(m) - 1;
                    break;
                }
            }
            const bool atEnd = d == N;
            const int64_t from = d - (atEnd ? 0 : b.traceBack + 1);
            if (lane == 0) {
                if (nBlocks < R.blockCap) {
                    BlockRec K;
                    K.region = r;
                    K.top = (int32_t) d;
                    K.T = (int32_t) T;
                    K.from = (int32_t) from;
                    K.cells = (int32_t) ((int64_t) dg[d + 1].coff - (int64_t) dg[T + 1].coff);
                    K.atEnd = atEnd;
                    K.decadeBase = 0;
                    bl[nBlocks] = K;
                } else {
                    err = 2;
                }
            }
            nBlocks++;
            /* total diagonals from, from-10, ... > T get their aux records, in that order */
            const int64_t nDec = (from - T + 9) / 10;
            for (int64_t j0 = 0; j0 < nDec; j0 += 32) {
                const int64_t j = j0 + lane;
                const int64_t dt = from - 10 * j;
                int64_t size = 0;
                if (j < nDec) size = (int64_t) (b.auxF + 1) * dg[dt].width + (dt + 1 <= d ? dg[dt + 1].width : 0);
                int64_t incl = size;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int64_t t = __shfl_up_sync(FULL, incl, o);
                    if (lane >= o) incl += t;
                }
                if (j < nDec) dg[dt].aoff = (uint32_t) (auxD + incl - size);
                auxD += __shfl_sync(FULL, incl, 31);
            }
            __syncwarp();
            T = from;
            if (atEnd) break;
        }
    }
    err = __reduce_max_sync(FULL, err);
    maxW = __reduce_max_sync(FULL, maxW);
    int msr = 1;
    __syncwarp();
    for (int k = lane; k < nStrips; k += 32) msr = max(msr, st[k].dLast - st[k].dFirst + 1);
    msr = __reduce_max_sync(FULL, msr);
    int sorted = 1;
    for (int k = 1 + lane; k < nStrips; k += 32) sorted &= st[k].dFirst >= st[k - 1].dFirst && st[k].dLast >= st[k - 1].dLast && st[k].dLast >= st[k].dFirst;
    sorted = __all_sync(FULL, sorted) && st[0].dLast >= st[0].dFirst;
    if (lane == 0) {
        R.stripsSorted = (uint8_t) sorted;
        R.cells = cellsBefore;
        R.auxDoubles = auxD;
        R.nBlocks = nBlocks;
        R.maxW = maxW;
        R.maxStripRange = msr;
        R.err = err;
        b.regions[r] = R;
    }
}

} /* namespace cpb */
