/*
 * engine.cu -- host orchestration of libcpecan_b200 (C-ABI in include/cpecan_b200.h).
 *
 * One batch run =
 *   k_split_flags + host : split every pair at large anchor gaps into regions (cpb_split_points; reference
 *          getPosteriorProbsWithBandingSplittingAlignmentsByLargeGaps, impl/pairwiseAligner.c:1273-1326)
 *   K1   : device band builder + traceback schedule, one small D2H of per-region sizes
 *   host : pack regions into chunks that fit the scratch budget, bucket work by band width
 *   per chunk: k_forward -> k_backward -> k_totals -> k_posterior (count, write) | k_expect
 * There is no CPU fallback anywhere in this file: without a CUDA device every entry point fails.
 */
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <chrono>
#include <atomic>
#include <thread>
#include <vector>

#include "cpecan_b200.h"
#include "internal.h"
#include "kernels.cuh"
#include "strip_kernels.cuh"
#include "narrow_kernels.cuh"
#include "anchor_kernels.cuh"
#include "decode_kernels.cuh"

using namespace cpb;

/* ------------------------------------------------------------------------------------------------ */
static thread_local char g_error[1024] = "";

extern "C" void cpb_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}
extern "C" const char *cpb_last_error(void) { return g_error; }
extern "C" const char *cpb_version(void) { return "cpecan_b200 0.1 (sm_100a)"; }

#define CUDA_TRY(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t e_ = (expr);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            cpb_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(e_), __FILE__, __LINE__, cudaGetErrorString(e_)); \
            return CPB_ERR_CUDA;                                                                         \
        }                                                                                                \
    } while (0)

/* Device allocations released by one batch are kept for the next (cudaMalloc / cudaFree of multi-GB buffers costs
 * hundreds of milliseconds per batch otherwise).  Best fit within 2x; everything is returned to the driver when the
 * context is destroyed or an allocation fails. */
/* Counts the calls that change how much device memory the driver has free (cudaMalloc / cudaFree made here): while it stands still, a
 * context's last answer from cudaMemGetInfo -- which costs ~12 ms once a few hundred buffers are live -- is still good. */
static std::atomic<uint64_t> g_allocEpoch{ 1 };

struct DevPool {
    struct Item {
        void *p;
        size_t cap;
    };
    std::vector<Item> items;
    void *take(size_t bytes, size_t *capOut) {
        int best = -1;
        for (int i = 0; i < (int) items.size(); i++) {
            if (items[i].cap >= bytes && items[i].cap <= 2 * bytes + (size_t(1) << 20) && (best < 0 || items[i].cap < items[best].cap)) best = i;
        }
        if (best < 0) return nullptr;
        void *p = items[best].p;
        *capOut = items[best].cap;
        items.erase(items.begin() + best);
        return p;
    }
    void give(void *p, size_t cap) { items.push_back({ p, cap }); }
    void drain() {
        for (auto &it : items) cudaFree(it.p);
        if (!items.empty()) g_allocEpoch++;
        items.clear();
    }
};

/* grow-only device buffer */
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    DevPool *pool = nullptr;
    int reserve(size_t bytes) {
        if (bytes <= cap) return CPB_OK;
        release();
        if (pool != nullptr && (p = pool->take(bytes, &cap)) != nullptr) return CPB_OK;
        g_allocEpoch++;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess && pool != nullptr) {
            (void) cudaGetLastError();
            pool->drain();
            e = cudaMalloc(&p, bytes);
        }
        if (e != cudaSuccess) {
            cpb_set_error("cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
            (void) cudaGetLastError();
            p = nullptr;
            return CPB_ERR_MEMORY;
        }
        cap = bytes;
        return CPB_OK;
    }
    void release() {
        if (p) {
            if (pool != nullptr) {
                pool->give(p, cap);
            } else {
                cudaFree(p);
                g_allocEpoch++;
            }
        }
        p = nullptr;
        cap = 0;
    }
    template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
    void adopt(DevBuf &other) { /* takes over other's allocation; this buffer must be empty */
        p = other.p;
        cap = other.cap;
        pool = other.pool;
        other.p = nullptr;
        other.cap = 0;
    }
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); } /* local buffers on error paths; owners that release explicitly leave nothing to do here */
};

/* ------------------------------------------------------------------------------------------------ */
/* page-locked host buffers handed out to batches (anchor staging) and taken back when the batch goes: pinning costs milliseconds per
 * 100 MB, so the buffers are kept */
struct PinnedPool {
    struct Item {
        void *p;
        size_t cap;
        bool inUse;
    };
    std::vector<Item> items;
    void *take(size_t bytes) {
        for (auto &it : items) {
            if (!it.inUse && it.cap >= bytes) {
                it.inUse = true;
                return it.p;
            }
        }
        for (auto &it : items) { /* grow an idle one rather than keep both */
            if (!it.inUse) {
                cudaFreeHost(it.p);
                it.p = nullptr;
                if (cudaHostAlloc(&it.p, bytes, cudaHostAllocDefault) != cudaSuccess) {
                    (void) cudaGetLastError();
                    it.p = nullptr;
                    it.cap = 0;
                    return nullptr;
                }
                it.cap = bytes;
                it.inUse = true;
                return it.p;
            }
        }
        Item it = { nullptr, bytes, true };
        if (cudaHostAlloc(&it.p, bytes, cudaHostAllocDefault) != cudaSuccess) {
            (void) cudaGetLastError();
            return nullptr;
        }
        items.push_back(it);
        return it.p;
    }
    void give(void *p) {
        for (auto &it : items) {
            if (it.p == p) it.inUse = false;
        }
    }
    void drain() {
        for (auto &it : items) {
            if (it.p) cudaFreeHost(it.p);
        }
        items.clear();
    }
};

/* A host table that travels to and from the device every run (region and block records): page-locked memory from the context's
 * pool, so that the copies are DMA transfers instead of the driver's staged pageable path (~3x slower for these 10-20 MB tables);
 * ordinary heap memory if page-locked memory cannot be had.  resize() does not keep the contents. */
template <class T> struct HostArray {
    T *p = nullptr;
    size_t n = 0, cap = 0;
    PinnedPool *pool = nullptr;
    bool pinned = false;
    HostArray() = default;
    HostArray(const HostArray &) = delete;
    HostArray &operator=(const HostArray &) = delete;
    ~HostArray() { release(); }
    void release() {
        if (p != nullptr) {
            if (pinned) pool->give(p);
            else free(p);
        }
        p = nullptr;
        n = cap = 0;
    }
    bool resize(size_t m) {
        if (m > cap) {
            PinnedPool *keep = pool;
            release();
            pool = keep;
            const size_t want = m + m / 8 + 16;
            p = pool != nullptr ? static_cast<T *>(pool->take(want * sizeof(T))) : nullptr;
            pinned = p != nullptr;
            if (p == nullptr) p = static_cast<T *>(malloc(want * sizeof(T)));
            if (p == nullptr) return false;
            cap = want;
        }
        n = m;
        return true;
    }
    void clear() { n = 0; }
    size_t size() const { return n; }
    bool empty() const { return n == 0; }
    T *data() { return p; }
    const T *data() const { return p; }
    T &operator[](size_t i) { return p[i]; }
    const T &operator[](size_t i) const { return p[i]; }
    T &back() { return p[n - 1]; }
    T *begin() { return p; }
    T *end() { return p + n; }
};

struct cpb_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool ownStream = false;
    size_t scratchBudget = 0;
    size_t freePlusScratch = 0;  /* cudaMemGetInfo's free bytes + the scratch buffer's, as of allocation epoch freeEpoch (0: never asked) */
    uint64_t freeEpoch = 0;
    DevBuf scratch;
    DevBuf boundary, counters, negRecord, progress; /* strip engine: per-warp-slot boundary rings, work-fetch counters, one LOG_ZERO ring record */
    DevBuf fixups;                                  /* posterior write pass: one counter (first 16 bytes), then PintFixup records */
    cudaStream_t copyStream = nullptr;              /* result sinks: device-to-host copies of finished chunks beside the next chunk's kernels */
    int smCount = 148;
    DevPool pool;              /* buffers handed back by destroyed batches */
    PinnedPool pinned;         /* page-locked host staging, same idea */
};

static const int kStripWPC = 4; /* warps per CTA of the strip kernels */
static const int kBwdWideBand = 1500; /* widest diagonal (cells) from which the backward kernel runs in its 3-CTAs-per-SM (168-register) build */
static const int64_t kSymPad = 64; /* bytes of 'n' before and after the symbol arrays */

static int configure_kernels() {
    const int maxSmem = 227 * 1024;
    CUDA_TRY(cudaFuncSetAttribute((const void *) k_expect<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxSmem));
    CUDA_TRY(cudaFuncSetAttribute((const void *) k_expect<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxSmem));
    return CPB_OK;
}

extern "C" int cpb_context_create(int device, void *stream, cpb_context **out) {
    if (out == nullptr) return CPB_ERR_ARGUMENT;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cpb_set_error("no CUDA device available (%s); libcpecan_b200 has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        (void) cudaGetLastError();
        return CPB_ERR_CUDA;
    }
    if (device < 0 || device >= count) {
        cpb_set_error("device %d out of range (have %d)", device, count);
        return CPB_ERR_ARGUMENT;
    }
    CUDA_TRY(cudaSetDevice(device));
    cpb_context *ctx = new cpb_context();
    ctx->device = device;
    if (stream != nullptr) {
        ctx->stream = (cudaStream_t) stream;
    } else {
        cudaError_t e2 = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        if (e2 != cudaSuccess) {
            cpb_set_error("cudaStreamCreate failed: %s", cudaGetErrorString(e2));
            delete ctx;
            return CPB_ERR_CUDA;
        }
        ctx->ownStream = true;
    }
    {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->smCount = prop.multiProcessorCount;
    }
    int rc = configure_kernels();
    if (rc == CPB_OK && (rc = ctx->negRecord.reserve(BND_REC * sizeof(double))) == CPB_OK) {
        double neg[BND_REC];
#ifdef CPB_FINITE_LOG_ZERO
        for (int i = 0; i < BND_REC; i++) neg[i] = -1e290; /* the kernels' LOG_ZERO stand-in (kernels.cuh) */
#else
        for (int i = 0; i < BND_REC; i++) neg[i] = -INFINITY;
#endif
        if (cudaMemcpy(ctx->negRecord.p, neg, sizeof(neg), cudaMemcpyHostToDevice) != cudaSuccess) {
            cpb_set_error("cudaMemcpy failed: %s", cudaGetErrorString(cudaGetLastError()));
            rc = CPB_ERR_CUDA;
        }
    }
    if (rc != CPB_OK) {
        if (ctx->ownStream) cudaStreamDestroy(ctx->stream);
        delete ctx;
        return rc;
    }
    *out = ctx;
    return CPB_OK;
}

extern "C" void cpb_context_destroy(cpb_context *ctx) {
    if (ctx == nullptr) return;
    cudaSetDevice(ctx->device);
    ctx->scratch.release();
    ctx->boundary.release();
    ctx->negRecord.release();
    ctx->progress.release();
    ctx->fixups.release();
    if (ctx->copyStream != nullptr) cudaStreamDestroy(ctx->copyStream);
    ctx->pool.drain();
    ctx->pinned.drain();
    ctx->counters.release();
    if (ctx->ownStream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

/* page-locked host memory from the context's pool (result staging of the host layer: a device-to-host copy into pageable memory runs at a
 * fraction of the link's rate) */
extern "C" void *cpb_pinned_alloc(cpb_context *ctx, size_t bytes) {
    if (ctx == nullptr) return nullptr;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return nullptr;
    return ctx->pinned.take(bytes > 0 ? bytes : 1);
}
extern "C" void cpb_pinned_free(cpb_context *ctx, void *p) {
    if (ctx != nullptr && p != nullptr) ctx->pinned.give(p);
}

extern "C" void cpb_context_set_scratch_budget(cpb_context *ctx, size_t bytes) {
    if (ctx) ctx->scratchBudget = bytes;
}

/* ------------------------------------------------------------------------------------------------ */
struct Chunk {
    int64_t region0, region1; /* [region0, region1) */
    int64_t block0, block1;   /* positions in the compact block order */
    int64_t cells, aux, maskWords, decades;
    int64_t stride;
    int64_t allBlocksOff;                /* offset of the chunk's in-order block list */
    int64_t stripFwdOff, stripBwdOff;    /* strip engine: regions / blocks sorted by cost */
    int64_t pair0, pair1;                /* pairs touched: [pair0, pair1] inclusive */
};

struct PlanKey { /* what a run's regions, bands, schedule, chunks and work lists depend on, apart from the batch itself */
    int64_t mode, states, split, expansion, dynamic, minDiags, traceBack, budget;
};

struct cpb_batch {
    cpb_context *ctx = nullptr;
    int64_t n = 0;
    std::vector<int64_t> xOff, yOff, aOff;
    int32_t *anchors = nullptr;      /* host copy of the anchor triples as the device has them (page-locked, from ctx->pinned) */
    std::vector<int32_t> anchorsOwn; /* fallback if page-locked memory cannot be had */
    std::vector<uint8_t> rl, rr;
    int32_t *sink[3] = { nullptr, nullptr, nullptr }; /* host buffers that receive the triples of each list while the run goes on */
    int64_t sinkCap[3] = { 0, 0, 0 };                 /* their capacity in triples */
    bool sunk[3] = { false, false, false };           /* the last run delivered the whole list into its sink */
    bool reweighted = false;         /* cpb_batch_reweight_pairs has rewritten list 0 of the last run in place */
    int64_t oddExpansionPair = -1;   /* first pair with an odd anchor expansion: only an error for runs with dynamicAnchorExpansion (:166) */
    DevBuf symX, symY, dAnchors;
    DevBuf keptX, keptY; /* the sequence bytes upper-cased (toupper): the decoders compare bytes, which the 0..4 symbols cannot */
    DevBuf dPairTab;   /* aOff, xOff, yOff as the device needs them for k_split_flags: 3 x (n + 1) int64 */
    DevBuf splitFlags; /* one bit per gap between anchors: 1 = getSplitPoints cuts the pair there; word 0 of the buffer counts the pairs with a cut */
    /* run state */
    DevBuf strips;
    DevBuf regions, diags, blocks, totals, lists, counts, offsets, masks, tileSums, pairCounts, partials, pairBlockOff, perPair, hmmTotal, forwardOut;
    DevBuf ckRegions, ckDiags, ckSizes, ckpt; /* two-pass forward: plane-less first pass over the regions, block checkpoints */
    DevBuf out[3];
    int64_t outCount[3] = { 0, 0, 0 };
    std::vector<int64_t> pairOff[3]; /* n+1 */
    /* the alignment list: one alignment per pair from the last decode call (cpb_batch_ordered_chain, cpb_batch_mea), cleared by every run */
    DevBuf aln;
    std::vector<int64_t> alnOff; /* n+1 */
    bool alnValid = false;
    int lastMode = -1, lastS = 0;
    CpbRunStats stats;
    HostArray<RegionDev> hRegions;
    HostArray<BlockRec> hBlocks; /* compact, region order */
    /* the plan of the last run, kept for the next one with the same key (run_impl) */
    std::vector<Chunk> chunks;
    PlanKey planKey;
    bool planValid = false;
    size_t planScratch = 0;
    CpbRunStats planStats;
};

static int find_anchors(cpb_batch *b, const CpbParams *p);

/* cpb_batch_create and cpb_batch_create_anchored: the caller's anchors, or (anchorParams != nullptr) those find_anchors makes on the
 * device from the raw sequences before they are encoded */
static int batch_create(cpb_context *ctx, int64_t nPairs, const char *seqX, const int64_t *xOff, const char *seqY, const int64_t *yOff,
                        const int64_t *anchors, const int64_t *anchorOff, const CpbParams *anchorParams, const uint8_t *raggedLeft,
                        const uint8_t *raggedRight, cpb_batch **out) {
    if (ctx == nullptr || out == nullptr || nPairs < 0 || xOff == nullptr || yOff == nullptr) {
        cpb_set_error("cpb_batch_create: bad argument");
        return CPB_ERR_ARGUMENT;
    }
    /* The kernels trust these arrays (region lengths and anchor coordinates are int32 on the device, the band builder's bisection
     * relies on x + y growing by at least 2 per anchor): everything the reference states as asserts (impl/pairwiseAligner.c:214-219)
     * is checked here, once, and reported with the index of the offending pair. */
    if (xOff[0] != 0 || yOff[0] != 0 || (anchorOff != nullptr && anchorOff[0] != 0)) {
        cpb_set_error("cpb_batch_create: offset arrays must start at 0");
        return CPB_ERR_ARGUMENT;
    }
    for (int64_t i = 0; i < nPairs; i++) {
        const int64_t lX = xOff[i + 1] - xOff[i], lY = yOff[i + 1] - yOff[i], nAi = anchorOff != nullptr ? anchorOff[i + 1] - anchorOff[i] : 0;
        if (lX < 0 || lY < 0 || nAi < 0 || lX + lY > (int64_t) 0x7FFFFF00) {
            cpb_set_error("cpb_batch_create: pair %lld: offsets are not non-decreasing, or the sequences are too long (lengths %lld, %lld, %lld anchors)",
                          (long long) i, (long long) lX, (long long) lY, (long long) nAi);
            return CPB_ERR_ARGUMENT;
        }
    }
    if ((xOff[nPairs] > 0 && seqX == nullptr) || (yOff[nPairs] > 0 && seqY == nullptr) || (anchorOff != nullptr && anchorOff[nPairs] > 0 && anchors == nullptr)) {
        cpb_set_error("cpb_batch_create: a sequence or anchor array is NULL although its offsets say it is not empty");
        return CPB_ERR_ARGUMENT;
    }
    *out = nullptr;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cpb_batch *b = new cpb_batch();
    b->ctx = ctx;
    b->hRegions.pool = &ctx->pinned;
    b->hBlocks.pool = &ctx->pinned;
    struct Guard { /* every early return below frees the batch, its device buffers and its page-locked anchor buffer */
        cpb_batch *b;
        ~Guard() {
            if (b != nullptr) cpb_batch_destroy(b);
        }
    } guard{ b };
    {
        DevBuf *all[] = { &b->strips, &b->symX, &b->symY, &b->dAnchors, &b->dPairTab, &b->splitFlags, &b->regions, &b->diags, &b->blocks, &b->totals, &b->lists, &b->counts, &b->offsets,
                          &b->masks, &b->tileSums, &b->pairCounts, &b->partials, &b->pairBlockOff, &b->perPair, &b->hmmTotal, &b->forwardOut, &b->out[0],
                          &b->out[1], &b->out[2], &b->ckRegions, &b->ckDiags, &b->ckSizes, &b->ckpt, &b->keptX, &b->keptY, &b->aln };
        for (DevBuf *d : all) d->pool = &ctx->pool;
    }
    b->n = nPairs;
    b->xOff.assign(xOff, xOff + nPairs + 1);
    b->yOff.assign(yOff, yOff + nPairs + 1);
    if (anchorOff != nullptr) b->aOff.assign(anchorOff, anchorOff + nPairs + 1);
    else b->aOff.assign(nPairs + 1, 0);
    const int64_t nA = b->aOff[nPairs];
    b->rl.assign(nPairs, 0);
    b->rr.assign(nPairs, 0);
    if (raggedLeft) b->rl.assign(raggedLeft, raggedLeft + nPairs);
    if (raggedRight) b->rr.assign(raggedRight, raggedRight + nPairs);
    memset(&b->stats, 0, sizeof(b->stats));

    const int64_t nx = xOff[nPairs], ny = yOff[nPairs];
    int rc = CPB_OK;
    /* the strip kernels index symbols up to 32 positions outside a region without bounds tests: pad both ends with 'n' */
    if ((rc = b->symX.reserve(nx + 2 * kSymPad)) != CPB_OK || (rc = b->symY.reserve(ny + 2 * kSymPad)) != CPB_OK ||
        (rc = b->keptX.reserve(std::max<int64_t>(nx, 1))) != CPB_OK || (rc = b->keptY.reserve(std::max<int64_t>(ny, 1))) != CPB_OK)
        return rc;
    cudaStream_t st = ctx->stream;
    CUDA_TRY(cudaMemsetAsync(b->symX.p, 4, nx + 2 * kSymPad, st));
    CUDA_TRY(cudaMemsetAsync(b->symY.p, 4, ny + 2 * kSymPad, st));
    if (nx > 0) CUDA_TRY(cudaMemcpyAsync(b->symX.as<uint8_t>() + kSymPad, seqX, nx, cudaMemcpyHostToDevice, st));
    if (ny > 0) CUDA_TRY(cudaMemcpyAsync(b->symY.as<uint8_t>() + kSymPad, seqY, ny, cudaMemcpyHostToDevice, st));
    if (anchorParams != nullptr) {
        if ((rc = find_anchors(b, anchorParams)) != CPB_OK) return rc; /* reads the raw bytes: the soft mask is their case */
    } else if ((rc = b->dAnchors.reserve(std::max<int64_t>(nA, 1) * 3 * sizeof(int32_t))) != CPB_OK) {
        return rc;
    }
    if (nx > 0) k_encode<<<(unsigned) ((nx + 255) / 256), 256, 0, st>>>(b->symX.as<uint8_t>() + kSymPad, b->keptX.as<uint8_t>(), nx);
    if (ny > 0) k_encode<<<(unsigned) ((ny + 255) / 256), 256, 0, st>>>(b->symY.as<uint8_t>() + kSymPad, b->keptY.as<uint8_t>(), ny);
    if (anchorParams == nullptr && nA > 0) {
        /* int64 triples of the caller -> int32 triples, straight into a page-locked buffer that serves both the copy to the device
         * and the host-side region construction of every run; a few host threads share the conversion */
        const size_t bytes = (size_t) (3 * nA) * sizeof(int32_t);
        b->anchors = static_cast<int32_t *>(ctx->pinned.take(bytes));
        if (b->anchors == nullptr) {
            b->anchorsOwn.resize((size_t) (3 * nA));
            b->anchors = b->anchorsOwn.data();
        }
        int32_t *dst = b->anchors;
        /* conversion and validation in one pass over the triples, pairs dealt to a few host threads in contiguous ranges */
        std::atomic<int64_t> badPair{ -1 }, oddPair{ -1 };
        auto convert = [&](int64_t p0, int64_t p1) {
            for (int64_t i = p0; i < p1; i++) {
                const int64_t lX = b->xOff[i + 1] - b->xOff[i], lY = b->yOff[i + 1] - b->yOff[i];
                int64_t px = -1, py = -1;
                bool ok = true, even = true;
                for (int64_t k = b->aOff[i]; k < b->aOff[i + 1]; k++) {
                    const int64_t x = anchors[3 * k], y = anchors[3 * k + 1], e = anchors[3 * k + 2];
                    ok &= x > px && y > py && x < lX && y < lY && e >= 0 && e <= 0x7FFFFFFF;
                    even &= (e & 1) == 0;
                    px = x;
                    py = y;
                    dst[3 * k] = (int32_t) x;
                    dst[3 * k + 1] = (int32_t) y;
                    dst[3 * k + 2] = (int32_t) e;
                }
                int64_t expect = -1;
                if (!ok) badPair.compare_exchange_strong(expect, i);
                expect = -1;
                if (!even) oddPair.compare_exchange_strong(expect, i);
            }
        };
        const int64_t nThreads = std::max<int64_t>(1, std::min<int64_t>({ (int64_t) std::thread::hardware_concurrency(), (int64_t) 8, (3 * nA) >> 20, nPairs }));
        if (nThreads <= 1) {
            convert(0, nPairs);
        } else {
            /* ranges of pairs holding about the same number of anchors */
            std::vector<std::thread> pool;
            int64_t p0 = 0;
            for (int64_t t = 0; t < nThreads; t++) {
                const int64_t want = nA * (t + 1) / nThreads;
                int64_t p1 = t + 1 == nThreads ? nPairs : (int64_t) (std::upper_bound(b->aOff.begin(), b->aOff.end(), want) - b->aOff.begin()) - 1;
                p1 = std::max(p0, std::min(p1, nPairs));
                pool.emplace_back(convert, p0, p1);
                p0 = p1;
            }
            for (auto &t : pool) t.join();
        }
        b->oddExpansionPair = oddPair.load();
        if (badPair.load() >= 0) {
            cpb_set_error("cpb_batch_create: pair %lld: anchors must be (x, y, expansion) with 0 <= x < lX, 0 <= y < lY, x and y strictly increasing and "
                          "expansion >= 0 (impl/pairwiseAligner.c:214-219)",
                          (long long) badPair.load());
            return CPB_ERR_ARGUMENT;
        }
        CUDA_TRY(cudaMemcpyAsync(b->dAnchors.p, b->anchors, bytes, cudaMemcpyHostToDevice, st));
    }
    if (nPairs > 0) {
        const size_t tab = (size_t) (nPairs + 1) * sizeof(int64_t);
        if ((rc = b->dPairTab.reserve(3 * tab)) != CPB_OK) return rc;
        CUDA_TRY(cudaMemcpyAsync(b->dPairTab.as<char>(), b->aOff.data(), tab, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(b->dPairTab.as<char>() + tab, b->xOff.data(), tab, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(b->dPairTab.as<char>() + 2 * tab, b->yOff.data(), tab, cudaMemcpyHostToDevice, st));
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    guard.b = nullptr;
    *out = b;
    return CPB_OK;
}

extern "C" int cpb_batch_create(cpb_context *ctx, int64_t nPairs, const char *seqX, const int64_t *xOff, const char *seqY, const int64_t *yOff,
                                const int64_t *anchors, const int64_t *anchorOff, const uint8_t *raggedLeft, const uint8_t *raggedRight,
                                cpb_batch **out) {
    return batch_create(ctx, nPairs, seqX, xOff, seqY, yOff, anchors, anchorOff, nullptr, raggedLeft, raggedRight, out);
}

extern "C" int cpb_batch_create_anchored(cpb_context *ctx, int64_t nPairs, const char *seqX, const int64_t *xOff, const char *seqY,
                                         const int64_t *yOff, const uint8_t *raggedLeft, const uint8_t *raggedRight, const CpbParams *p,
                                         cpb_batch **out) {
    if (p == nullptr || p->constraintDiagonalTrim < 0 || p->diagonalExpansion < 0 || p->diagonalExpansion > 0x7FFFFFFF) {
        cpb_set_error("cpb_batch_create_anchored: %s", p == nullptr ? "no parameters" : "constraintDiagonalTrim and diagonalExpansion must be in [0, 2^31)");
        return CPB_ERR_ARGUMENT;
    }
    return batch_create(ctx, nPairs, seqX, xOff, seqY, yOff, nullptr, nullptr, p, raggedLeft, raggedRight, out);
}

extern "C" int64_t cpb_batch_anchor_count(const cpb_batch *b) { return b != nullptr ? b->aOff[b->n] : 0; }

extern "C" int cpb_batch_fetch_anchors(const cpb_batch *b, int64_t *offsets, int64_t *triples) {
    if (b == nullptr || offsets == nullptr || (triples == nullptr && b->aOff[b->n] > 0)) {
        cpb_set_error("cpb_batch_fetch_anchors: bad argument");
        return CPB_ERR_ARGUMENT;
    }
    memcpy(offsets, b->aOff.data(), (size_t) (b->n + 1) * sizeof(int64_t));
    for (int64_t k = 0; k < 3 * b->aOff[b->n]; k++) triples[k] = b->anchors[k];
    return CPB_OK;
}

extern "C" void cpb_batch_destroy(cpb_batch *b) {
    if (b == nullptr) return;
    cudaSetDevice(b->ctx->device);
    DevBuf *bufs[] = { &b->strips, &b->symX, &b->symY, &b->dAnchors, &b->dPairTab, &b->splitFlags, &b->regions, &b->diags, &b->blocks, &b->totals, &b->lists, &b->counts,
                       &b->offsets, &b->masks, &b->tileSums, &b->pairCounts, &b->partials, &b->pairBlockOff, &b->perPair, &b->hmmTotal, &b->forwardOut, &b->out[0], &b->out[1],
                       &b->out[2], &b->ckRegions, &b->ckDiags, &b->ckSizes, &b->ckpt, &b->keptX, &b->keptY, &b->aln };
    for (DevBuf *d : bufs) d->release();
    if (b->anchors != nullptr && b->anchorsOwn.empty()) b->ctx->pinned.give(b->anchors);
    delete b;
}

/* ------------------------------------------------------------------------------------------------
 * anchors on the device (anchor_kernels.cuh): getBlastPairsForPairwiseAlignmentParameters of host/anchors.c for every pair at once
 * ---------------------------------------------------------------------------------------------- */
/* word_length of anchors.c: the smallest k in 11..24 with 4^k >= 64 max(lX, lY) */
static int anchor_word_length(int64_t lX, int64_t lY) {
    int k = 11;
    double space = 4194304.0; /* 4^11 */
    while (k < 24 && space < 64.0 * (double) (lX < lY ? lY : lX)) {
        k++;
        space *= 4.0;
    }
    return k;
}

/* exclusive scan of n int32 counts into offsets[0..n], offsets[n] = startAt + the sum (tiles: (n + SCAN_TILE - 1) / SCAN_TILE entries) */
static void scan_counts(cudaStream_t st, const int32_t *counts, int64_t n, int64_t startAt, int64_t *tiles, int64_t *offsets) {
    const int64_t nTiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    if (nTiles > 0) k_scan_tiles<<<(unsigned) nTiles, 256, 0, st>>>(counts, n, tiles);
    k_scan_sums<<<1, 1, 0, st>>>(tiles, nTiles, startAt, offsets + n);
    if (nTiles > 0) k_scan_apply<<<(unsigned) nTiles, 256, 0, st>>>(counts, n, tiles, offsets);
}

static unsigned grid_of(int64_t n, int threads) { return (unsigned) std::max<int64_t>(1, (n + threads - 1) / threads); }

/* Scratch bytes of one problem: its k-mer table, 40 bytes per X position (hit, seed flag, seed offset, seed, chain arrays), 8 per Y
 * position (the Fenwick tree) and its records. */
static size_t anchor_problem_bytes(int64_t lX, int64_t lY, int64_t tableEntries) {
    return (size_t) (16 * tableEntries + 40 * lX + 8 * (lY + 2) + sizeof(AnchorProblem) + 64);
}

/* Every problem's anchors: triples into tri (capacity: the problems' lX summed), problem p's at [off[p], off[p + 1]).  probs holds the
 * problems' x, y, lX, lY, mask, dx, dy; the rest is filled in here.  The problems go through the kernels in chunks whose scratch fits the
 * context's budget. */
static int anchor_problems(cpb_batch *b, std::vector<AnchorProblem> &probs, const CpbParams *p, DevBuf &tri, DevBuf &off, int64_t *total) {
    cpb_context *ctx = b->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t nP = (int64_t) probs.size();
    int64_t bound = 0;
    for (AnchorProblem &P : probs) bound += P.lX;
    int rc;
    if ((rc = tri.reserve((size_t) std::max<int64_t>(bound, 1) * 3 * sizeof(int32_t))) != CPB_OK ||
        (rc = off.reserve((size_t) (nP + 1) * sizeof(int64_t))) != CPB_OK)
        return rc;
    size_t budget = ctx->scratchBudget;
    if (budget == 0) {
        size_t freeB = 0, totalB = 0;
        CUDA_TRY(cudaMemGetInfo(&freeB, &totalB));
        budget = (size_t) ((double) (freeB + ctx->scratch.cap) * 0.70);
    }
    const size_t fixed = 16 * 256; /* alignment of the chunk's arrays */
    int64_t running = 0;
    for (int64_t p0 = 0; p0 < nP;) {
        int64_t p1 = p0, X = 0, Y = 0, E = 0;
        size_t bytes = fixed;
        while (p1 < nP) {
            AnchorProblem &P = probs[(size_t) p1];
            int64_t cap = 16;
            while (cap < 2 * (int64_t) P.lY) cap <<= 1;
            const size_t need = anchor_problem_bytes(P.lX, P.lY, cap);
            if (fixed + need > budget) {
                cpb_set_error("anchoring a %d x %d problem needs %zu bytes of scratch, more than the budget of %zu", P.lX, P.lY, fixed + need, budget);
                return CPB_ERR_MEMORY;
            }
            if (bytes + need > budget || p1 - p0 >= (1 << 30)) break;
            bytes += need;
            P.k = anchor_word_length(P.lX, P.lY);
            P.capMask = (int32_t) (cap - 1);
            P.xPos = X;
            P.yPos = Y;
            P.tab = E;
            X += P.lX;
            Y += P.lY + 2;
            E += cap;
            p1++;
        }
        const int nC = (int) (p1 - p0);
        /* the chunk's arrays, 256-byte aligned, in ctx->scratch */
        size_t at = 0;
        auto carve = [&](size_t n) {
            const size_t here = at;
            at += (n + 255) & ~(size_t) 255;
            return here;
        };
        const size_t oDesc = carve(nC * sizeof(AnchorProblem)), oTab = carve(E * sizeof(KmerEntry)), oHit = carve(X * 4), oFlag = carve(X * 4),
                     oSeedOff = carve((X + 1) * 8), oSeeds = carve(X * sizeof(int3)), oScore = carve(X * 4), oPrev = carve(X * 4), oOrder = carve(X * 4),
                     oFenS = carve(Y * 4), oFenW = carve(Y * 4), oChain = carve(nC * 4), oCount = carve(nC * 4),
                     oTiles = carve(((std::max(X, (int64_t) nC) + SCAN_TILE - 1) / SCAN_TILE + 1) * 8);
        if ((rc = ctx->scratch.reserve(std::max<size_t>(at, 256))) != CPB_OK) return rc;
        char *s = ctx->scratch.as<char>();
        AnchorProblem *dP = reinterpret_cast<AnchorProblem *>(s + oDesc);
        KmerEntry *dTab = reinterpret_cast<KmerEntry *>(s + oTab);
        int32_t *dHit = reinterpret_cast<int32_t *>(s + oHit), *dFlag = reinterpret_cast<int32_t *>(s + oFlag);
        int64_t *dSeedOff = reinterpret_cast<int64_t *>(s + oSeedOff), *dTiles = reinterpret_cast<int64_t *>(s + oTiles);
        int3 *dSeeds = reinterpret_cast<int3 *>(s + oSeeds);
        int32_t *dScore = reinterpret_cast<int32_t *>(s + oScore), *dPrev = reinterpret_cast<int32_t *>(s + oPrev), *dOrder = reinterpret_cast<int32_t *>(s + oOrder);
        int32_t *dFenS = reinterpret_cast<int32_t *>(s + oFenS), *dFenW = reinterpret_cast<int32_t *>(s + oFenW);
        int32_t *dChain = reinterpret_cast<int32_t *>(s + oChain), *dCount = reinterpret_cast<int32_t *>(s + oCount);
        const uint8_t *sx = b->symX.as<uint8_t>(), *sy = b->symY.as<uint8_t>();
        int64_t *dOff = off.as<int64_t>() + p0;
        CUDA_TRY(cudaMemcpyAsync(dP, probs.data() + p0, nC * sizeof(AnchorProblem), cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemsetAsync(dTab, 0xFF, E * sizeof(KmerEntry), st));
        CUDA_TRY(cudaMemsetAsync(dFenS, 0, Y * 4, st));
        CUDA_TRY(cudaMemsetAsync(dFenW, 0, Y * 4, st));
        k_anchor_index<<<grid_of(Y, 256), 256, 0, st>>>(dP, nC, Y, sy, dTab);
        k_anchor_hits<<<grid_of(X, 256), 256, 0, st>>>(dP, nC, X, sx, dTab, dHit);
        k_anchor_seed_flags<<<grid_of(X, 256), 256, 0, st>>>(dP, nC, X, dHit, dFlag);
        scan_counts(st, dFlag, X, 0, dTiles, dSeedOff);
        k_anchor_seeds<<<grid_of(X, 256), 256, 0, st>>>(dP, nC, X, dHit, dFlag, dSeedOff, dSeeds);
        k_anchor_chain<<<grid_of(nC, 64), 64, 0, st>>>(dP, nC, sx, sy, dSeedOff, dSeeds, dScore, dPrev, dOrder, dFenS, dFenW, p->constraintDiagonalTrim,
                                                       dChain, dCount);
        scan_counts(st, dCount, nC, running, dTiles, dOff);
        k_anchor_runs<<<grid_of(nC, 64), 64, 0, st>>>(dP, nC, sx, sy, dSeedOff, dSeeds, dOrder, dChain, p->constraintDiagonalTrim,
                                                      (int32_t) p->diagonalExpansion, dOff, tri.as<int32_t>());
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(&running, dOff + nC, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st)); /* the next chunk's scan starts from this total, and reuses the scratch */
        p0 = p1;
    }
    if (nP == 0) CUDA_TRY(cudaMemsetAsync(off.p, 0, sizeof(int64_t), st));
    *total = running;
    return CPB_OK;
}

/* getBlastPairsForPairwiseAlignmentParameters (anchors.c:361-381) of every pair: level 1 on every matrix bigger than
 * anchorMatrixBiggerThanThis, level 2 on every gap of those lists that is still that big, merged per pair.  The lists need no sort and
 * no overlap filter: a chain's triples ascend strictly in x and y, and a gap's lie strictly inside it.  Fills b->aOff, b->anchors (one
 * copy back), b->dAnchors and b->oddExpansionPair.  The per-position arrays come out of the scratch budget; the lists and the per-gap
 * tables, which grow with the anchors, are batch buffers like the anchors themselves. */
static int find_anchors(cpb_batch *b, const CpbParams *p) {
    cpb_context *ctx = b->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = b->n;
    std::vector<AnchorProblem> l1;
    std::vector<int32_t> problemOf((size_t) std::max<int64_t>(n, 1), -1), pairOf, lX1, lY1;
    for (int64_t i = 0; i < n; i++) {
        const int64_t lX = b->xOff[i + 1] - b->xOff[i], lY = b->yOff[i + 1] - b->yOff[i];
        if (lX * lY <= p->anchorMatrixBiggerThanThis) continue;
        AnchorProblem P;
        memset(&P, 0, sizeof(P));
        P.x = kSymPad + b->xOff[i];
        P.y = kSymPad + b->yOff[i];
        P.lX = (int32_t) lX;
        P.lY = (int32_t) lY;
        P.mask = 1;
        problemOf[(size_t) i] = (int32_t) l1.size();
        pairOf.push_back((int32_t) i);
        lX1.push_back(P.lX);
        lY1.push_back(P.lY);
        l1.push_back(P);
    }
    const int64_t nP = (int64_t) l1.size();
    DevBuf tri1, off1, tri2, off2, tab, flags, gapIdx, gaps, sizes, slotPos, tiles, counts, aOffDev;
    DevBuf *all[] = { &tri1, &off1, &tri2, &off2, &tab, &flags, &gapIdx, &gaps, &sizes, &slotPos, &tiles, &counts, &aOffDev };
    for (DevBuf *d : all) d->pool = &ctx->pool;
    int rc;
    int64_t n1 = 0, n2 = 0;
    if ((rc = anchor_problems(b, l1, p, tri1, off1, &n1)) != CPB_OK) return rc;
    /* level 2: gap slot off1[q] + q + g is gap g of problem q */
    const int64_t nSlots = n1 + nP;
    const size_t tabBytes = (size_t) (3 * nP + n + 3) * sizeof(int32_t);
    if ((rc = tab.reserve(tabBytes)) != CPB_OK || (rc = flags.reserve((size_t) (nSlots + 1) * 4)) != CPB_OK ||
        (rc = gapIdx.reserve((size_t) (nSlots + 1) * 8)) != CPB_OK || (rc = sizes.reserve((size_t) (nSlots + 1) * 4)) != CPB_OK ||
        (rc = slotPos.reserve((size_t) (nSlots + 1) * 8)) != CPB_OK ||
        (rc = tiles.reserve((size_t) ((std::max(nSlots, n) + SCAN_TILE - 1) / SCAN_TILE + 1) * 8)) != CPB_OK ||
        (rc = counts.reserve((size_t) (n + 1) * 4)) != CPB_OK)
        return rc;
    int32_t *dLX = tab.as<int32_t>(), *dLY = dLX + nP, *dPairOf = dLY + nP, *dProblemOf = dPairOf + nP;
    if (nP > 0) {
        CUDA_TRY(cudaMemcpyAsync(dLX, lX1.data(), nP * 4, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(dLY, lY1.data(), nP * 4, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(dPairOf, pairOf.data(), nP * 4, cudaMemcpyHostToDevice, st));
    }
    if (n > 0) CUDA_TRY(cudaMemcpyAsync(dProblemOf, problemOf.data(), n * 4, cudaMemcpyHostToDevice, st));
    const int64_t *dOff1 = off1.as<int64_t>();
    const int32_t *dTri1 = tri1.as<int32_t>();
    int64_t nGaps = 0;
    if (nSlots > 0) {
        k_anchor_gap_flags<<<grid_of(nSlots, 256), 256, 0, st>>>((int) nP, dOff1, dTri1, dLX, dLY, nSlots, (long long) p->anchorMatrixBiggerThanThis,
                                                               flags.as<int32_t>());
        scan_counts(st, flags.as<int32_t>(), nSlots, 0, tiles.as<int64_t>(), gapIdx.as<int64_t>());
        CUDA_TRY(cudaMemcpyAsync(&nGaps, gapIdx.as<int64_t>() + nSlots, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    if (nGaps > 0) {
        if ((rc = gaps.reserve((size_t) nGaps * sizeof(AnchorGap))) != CPB_OK) return rc;
        k_anchor_gap_list<<<grid_of(nSlots, 256), 256, 0, st>>>((int) nP, dOff1, dTri1, dLX, dLY, dPairOf, nSlots, (long long) p->repeatMaskMatrixBiggerThanThis,
                                                              flags.as<int32_t>(), gapIdx.as<int64_t>(), gaps.as<AnchorGap>());
        std::vector<AnchorGap> hGaps((size_t) nGaps);
        CUDA_TRY(cudaMemcpyAsync(hGaps.data(), gaps.p, (size_t) nGaps * sizeof(AnchorGap), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        std::vector<AnchorProblem> l2((size_t) nGaps);
        for (int64_t q = 0; q < nGaps; q++) {
            const AnchorGap &G = hGaps[(size_t) q];
            AnchorProblem &P = l2[(size_t) q];
            memset(&P, 0, sizeof(P));
            P.x = kSymPad + b->xOff[G.pair] + G.x;
            P.y = kSymPad + b->yOff[G.pair] + G.y;
            P.lX = G.lX;
            P.lY = G.lY;
            P.mask = G.mask;
            P.dx = G.x;
            P.dy = G.y;
        }
        if ((rc = anchor_problems(b, l2, p, tri2, off2, &n2)) != CPB_OK) return rc;
    }
    /* merge: every gap slot's position in the final lists, then both levels' triples to their places */
    const int64_t nA = n1 + n2;
    if ((rc = b->dAnchors.reserve((size_t) std::max<int64_t>(nA, 1) * 3 * sizeof(int32_t))) != CPB_OK) return rc;
    int32_t *dOut = b->dAnchors.as<int32_t>();
    if (nSlots > 0) {
        k_anchor_slot_sizes<<<grid_of(nSlots, 256), 256, 0, st>>>((int) nP, dOff1, nSlots, flags.as<int32_t>(), gapIdx.as<int64_t>(), off2.as<int64_t>(),
                                                                sizes.as<int32_t>());
        scan_counts(st, sizes.as<int32_t>(), nSlots, 0, tiles.as<int64_t>(), slotPos.as<int64_t>());
        k_anchor_merge_level1<<<grid_of(nSlots, 256), 256, 0, st>>>((int) nP, dOff1, dTri1, nSlots, flags.as<int32_t>(), gapIdx.as<int64_t>(),
                                                                  off2.as<int64_t>(), slotPos.as<int64_t>(), dOut);
        if (n2 > 0)
            k_anchor_merge_level2<<<grid_of(n2, 256), 256, 0, st>>>((int) nGaps, gaps.as<AnchorGap>(), off2.as<int64_t>(), tri2.as<int32_t>(),
                                                                  slotPos.as<int64_t>(), dOut);
    }
    b->aOff.assign((size_t) n + 1, 0);
    if (n > 0) {
        if (nP > 0) {
            k_anchor_pair_counts<<<grid_of(n, 256), 256, 0, st>>>((int) n, dProblemOf, dOff1, slotPos.as<int64_t>(), counts.as<int32_t>());
        } else {
            CUDA_TRY(cudaMemsetAsync(counts.p, 0, (size_t) n * 4, st));
        }
        if ((rc = aOffDev.reserve((size_t) (n + 1) * 8)) != CPB_OK) return rc;
        scan_counts(st, counts.as<int32_t>(), n, 0, tiles.as<int64_t>(), aOffDev.as<int64_t>());
        CUDA_TRY(cudaMemcpyAsync(b->aOff.data(), aOffDev.p, (size_t) (n + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    }
    if (nA > 0) {
        const size_t bytes = (size_t) (3 * nA) * sizeof(int32_t);
        b->anchors = static_cast<int32_t *>(ctx->pinned.take(bytes));
        if (b->anchors == nullptr) {
            b->anchorsOwn.resize((size_t) (3 * nA));
            b->anchors = b->anchorsOwn.data();
        }
        CUDA_TRY(cudaMemcpyAsync(b->anchors, dOut, bytes, cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));
    if (p->diagonalExpansion & 1) {
        for (int64_t i = 0; i < n && b->oddExpansionPair < 0; i++)
            if (b->aOff[(size_t) i + 1] > b->aOff[(size_t) i]) b->oddExpansionPair = i;
    }
    return CPB_OK;
}

/* ------------------------------------------------------------------------------------------------
 * region construction on the host
 * ---------------------------------------------------------------------------------------------- */
/* Region records of every pair from the gaps k_split_flags marked (getSplitPoints, impl/pairwiseAligner.c:1230-1257; the model.c
 * restatement cpb_split_points is what the tests compare with).  `flags` = the host copy of the bit array, nullptr if no pair is cut
 * (or the mode never cuts: computeForwardProbability takes the whole matrix). */
static int build_regions(cpb_batch *b, const CpbParams *p, int mode, const uint32_t *flags) {
    /* Pairs are independent: every host thread of a pool makes the region records of a contiguous range of pairs with the offsets
     * into the device arrays counted from the start of its range; the ranges' totals are then prefix-summed and every thread moves its
     * records to their place in the batch's table.  A region's anchors are those between the two cuts that bound it, so nobody
     * walks the anchors here. */
    const int64_t n = b->n;
    struct Part {
        std::vector<RegionDev> regs;
        int64_t diags = 0, blocks = 0, strips = 0; /* totals of the range */
    };
    const int64_t nThreads = std::max<int64_t>(1, std::min<int64_t>({ (int64_t) std::thread::hardware_concurrency(), (int64_t) 16, n / 256 }));
    std::vector<Part> parts((size_t) nThreads);
    const int64_t half = (int64_t) sqrt((double) p->splitMatrixBiggerThanThis);
    auto work = [&](int64_t t) {
        const int64_t i0 = n * t / nThreads, i1 = n * (t + 1) / nThreads;
        Part &part = parts[(size_t) t];
        part.regs.reserve((size_t) (i1 - i0) + 16);
        for (int64_t i = i0; i < i1; i++) {
            const int64_t lX = b->xOff[i + 1] - b->xOff[i], lY = b->yOff[i + 1] - b->yOff[i];
            const int64_t a0 = b->aOff[i], nA = b->aOff[i + 1] - a0;
            const int32_t *an = b->anchors + 3 * a0;
            const size_t firstOfPair = part.regs.size();
            auto emit = [&](int64_t x1, int64_t y1, int64_t x2, int64_t y2, int64_t j0, int64_t j1) {
                RegionDev R;
                memset(&R, 0, sizeof(R));
                R.xBase = b->xOff[i] + x1;
                R.yBase = b->yOff[i] + y1;
                R.anchorBase = a0 + j0;
                R.nAnchors = (int32_t) (j1 - j0); /* the anchors before the region's last diagonal (impl/pairwiseAligner.c:1296-1308): those up to the cut */
                R.lX = (int32_t) (x2 - x1);
                R.lY = (int32_t) (y2 - y1);
                R.pair = (int32_t) i;
                R.ox = (int32_t) x1;
                R.oy = (int32_t) y1;
                /* consecutive traceback points are at least minDiags - (traceBack+1) diagonals apart (T moves to d - traceBack - 1) */
                R.blockCap = (int32_t) (((int64_t) R.lX + R.lY) / (p->minDiagsBetweenTraceBack - p->traceBackDiagonals - 1) + 2);
                R.diagBase = part.diags;
                R.blockBase = part.blocks;
                R.stripBase = part.strips;
                part.strips += (R.lX >> 5) + 1;
                part.diags += (int64_t) R.lX + R.lY + 3; /* lX+lY+1 diagonals and two sentinels */
                part.blocks += R.blockCap;
                part.regs.push_back(R);
            };
            int64_t openX = 0, openY = 0, openJ = 0; /* start of the region being grown, its first anchor */
            bool lastGapSplit = false;
            if (flags != nullptr && mode != CPB_MODE_FORWARD) {
                /* the set bits of [bit0, bit0 + nA], in ascending order */
                const int64_t bit0 = a0 + i, bit1 = bit0 + nA;
                for (int64_t w = bit0 >> 5; w <= bit1 >> 5; w++) {
                    uint32_t m = flags[w];
                    if (w == bit0 >> 5) m &= 0xFFFFFFFFu << (bit0 & 31);
                    if (w == bit1 >> 5 && (bit1 & 31) != 31) m &= (2u << (bit1 & 31)) - 1u;
                    while (m != 0) {
                        const int64_t g = (w << 5) + __builtin_ctz(m) - bit0;
                        m &= m - 1;
                        const int64_t prevX = g > 0 ? (int64_t) an[3 * (g - 1)] + 1 : 0, prevY = g > 0 ? (int64_t) an[3 * (g - 1) + 1] + 1 : 0;
                        const int64_t nextX = g < nA ? (int64_t) an[3 * g] : lX, nextY = g < nA ? (int64_t) an[3 * g + 1] : lY;
                        const int64_t gapX = nextX - prevX, gapY = nextY - prevY;
                        const int64_t hX = gapX / 2 > half ? half : gapX / 2, hY = gapY / 2 > half ? half : gapY / 2;
                        if (!(b->rl[i] && g == 0)) emit(openX, openY, prevX + hX, prevY + hY, openJ, g); /* a ragged left end drops the region before the first anchor */
                        openX = nextX - hX;
                        openY = nextY - hY;
                        openJ = g;
                        lastGapSplit = g == nA;
                    }
                }
            }
            if (!lastGapSplit || !b->rr[i]) emit(openX, openY, lX, lY, openJ, nA); /* a ragged right end drops the region after a trailing cut */
            const size_t nOfPair = part.regs.size() - firstOfPair;
            for (size_t r = 0; r < nOfPair; r++) {
                RegionDev &R = part.regs[firstOfPair + r];
                if (mode == CPB_MODE_FORWARD) {
                    R.raggedL = b->rl[i];
                    R.raggedR = b->rr[i];
                } else {
                    R.raggedL = b->rl[i] || r > 0;
                    R.raggedR = b->rr[i] || r + 1 < nOfPair;
                }
            }
        }
    };
    auto run_pool = [&](auto &&fn) {
        if (nThreads <= 1) {
            fn((int64_t) 0);
        } else {
            std::vector<std::thread> pool;
            for (int64_t t = 0; t < nThreads; t++) pool.emplace_back(fn, t);
            for (auto &t : pool) t.join();
        }
    };
    run_pool(work);
    std::vector<int64_t> first((size_t) nThreads + 1, 0), diag0((size_t) nThreads, 0), block0((size_t) nThreads, 0), strip0((size_t) nThreads, 0);
    int64_t diagBase = 0, blockBase = 0, stripBase = 0;
    for (int64_t t = 0; t < nThreads; t++) {
        first[(size_t) t + 1] = first[(size_t) t] + (int64_t) parts[(size_t) t].regs.size();
        diag0[(size_t) t] = diagBase;
        block0[(size_t) t] = blockBase;
        strip0[(size_t) t] = stripBase;
        diagBase += parts[(size_t) t].diags;
        blockBase += parts[(size_t) t].blocks;
        stripBase += parts[(size_t) t].strips;
    }
    if (!b->hRegions.resize((size_t) first[(size_t) nThreads])) {
        cpb_set_error("out of host memory for %lld region records", (long long) first[(size_t) nThreads]);
        return CPB_ERR_MEMORY;
    }
    run_pool([&](int64_t t) {
        RegionDev *out = b->hRegions.data() + first[(size_t) t];
        for (const RegionDev &R0 : parts[(size_t) t].regs) {
            RegionDev R = R0;
            R.diagBase += diag0[(size_t) t];
            R.blockBase += block0[(size_t) t];
            R.stripBase += strip0[(size_t) t];
            *out++ = R;
        }
    });
    return CPB_OK;
}

/* The smallest log-probability lp with exp(lp) >= threshold under THIS host's libm -- the reference decides p >= threshold with
 * p = exp(lp) from libm (impl/pairwiseAligner.c:656, :680), so comparing lp against this value on the device gives the reference's
 * keep decision exactly, whatever the device's own exp does in the last place.  Bisection over the doubles (libm's exp is monotone
 * around the crossing; that is verified for the 64 doubles on either side and reported if it ever fails). */
static double log_threshold_for_host_libm(double threshold) {
    if (!(threshold > 0.0)) return -INFINITY; /* p >= 0 holds for every cell, also for p = exp(LOG_ZERO) = 0 */
    auto key = [](double v) { /* order-preserving map of doubles to int64 */
        int64_t k;
        memcpy(&k, &v, sizeof(k));
        return k < 0 ? (int64_t) 0x8000000000000000ull - k : k;
    };
    auto unkey = [](int64_t k) {
        if (k < 0) k = (int64_t) 0x8000000000000000ull - k;
        double v;
        memcpy(&v, &k, sizeof(v));
        return v;
    };
    int64_t lo = key(-800.0), hi = key(1.0); /* exp(lo) = 0 < threshold <= 1 < exp(hi) */
    if (exp(unkey(hi)) < threshold) return INFINITY;
    while ((uint64_t) hi - (uint64_t) lo > 1) { /* as unsigned: hi - lo does not fit an int64 */
        const int64_t mid = (lo >> 1) + (hi >> 1) + (lo & hi & 1); /* hi - lo does not fit an int64 */
        if (exp(unkey(mid)) >= threshold) hi = mid;
        else lo = mid;
    }
    for (int k = 1; k <= 64; k++) {
        if (exp(unkey(hi + k)) < threshold || exp(unkey(hi - k)) >= threshold) {
            static bool warned = false;
            if (!warned) fprintf(stderr, "cpecan_b200: libm exp is not monotone around log(%.17g); posterior keep decisions next to the threshold may differ from the reference by one cell\n", threshold);
            warned = true;
            break;
        }
    }
    return unkey(hi);
}

static int check_params(const CpbParams *p) {
    /* the reference's preconditions, impl/pairwiseAligner.c:761-765 */
    if (p->traceBackDiagonals < 1 || p->diagonalExpansion < 0 || p->diagonalExpansion % 2 != 0 || p->minDiagsBetweenTraceBack < 2 ||
        p->traceBackDiagonals + 1 >= p->minDiagsBetweenTraceBack) {
        cpb_set_error("invalid PairwiseAlignmentParameters: traceBackDiagonals %lld, diagonalExpansion %lld, minDiagsBetweenTraceBack %lld",
                      (long long) p->traceBackDiagonals, (long long) p->diagonalExpansion, (long long) p->minDiagsBetweenTraceBack);
        return CPB_ERR_ARGUMENT;
    }
    if (!(p->threshold >= 0.0 && p->threshold <= 1.0)) {
        cpb_set_error("threshold %g outside [0,1]", p->threshold);
        return CPB_ERR_ARGUMENT;
    }
    return CPB_OK;
}

/* Orders idx[0..n) by cost, most expensive first, to within 1/1024 of the largest cost: a counting sort on the leading bits.  The
 * work-fetch order only needs the big items early; an exact std::sort of a few hundred thousand items was the largest host stage. */
template <class Cost> static void order_by_cost_descending(int32_t *idx, int64_t n, Cost cost) {
    if (n < 2) return;
    std::vector<int64_t> c((size_t) n); /* the costs, fetched once: the records they come from are 40 to 144 bytes apart */
    int64_t largest = 1;
    for (int64_t i = 0; i < n; i++) {
        c[(size_t) i] = cost(idx[i]);
        largest = std::max<int64_t>(largest, c[(size_t) i]);
    }
    int shift = 0;
    while ((largest >> shift) >= 2048) shift++;
    std::vector<int64_t> start(2049, 0);
    for (int64_t i = 0; i < n; i++) start[(size_t) (2047 - (c[(size_t) i] >> shift) + 1)]++;
    for (int k = 0; k < 2048; k++) start[k + 1] += start[k];
    std::vector<int32_t> out((size_t) n);
    for (int64_t i = 0; i < n; i++) out[(size_t) start[(size_t) (2047 - (c[(size_t) i] >> shift))]++] = idx[i];
    memcpy(idx, out.data(), (size_t) n * sizeof(int32_t));
}

struct EventPair {
    cudaEvent_t a, b;
    double *sink;
};

/* ------------------------------------------------------------------------------------------------ */
template <int S>
static int run_impl(cpb_batch *b, const CpbModel *m, const CpbParams *p, int mode) {
    cpb_context *ctx = b->ctx;
    cudaStream_t st = ctx->stream;
    CpbRunStats &stx = b->stats;
    memset(&stx, 0, sizeof(stx));
#ifdef CPB_FINITE_LOG_ZERO
    /* log(0) entries of the model (start / end vectors, impossible transitions of a loaded Hmm) become the kernels' finite stand-in */
    CpbModel finiteModel = *m;
    {
        double *groups[] = { finiteModel.start, finiteModel.raggedStart, finiteModel.end, finiteModel.raggedEnd, finiteModel.tLower, finiteModel.tMiddle,
                             finiteModel.tUpper, finiteModel.eMatch, finiteModel.eGapX, finiteModel.eGapY };
        const int sizes[] = { 5, 5, 5, 5, 4, 5, 4, 25, 5, 5 };
        for (int g = 0; g < 10; g++) {
            for (int i = 0; i < sizes[g]; i++) {
                if (!(groups[g][i] > -1e290)) groups[g][i] = -1e290;
            }
        }
    }
    m = &finiteModel;
#endif
    stx.nPairs = b->n;
    b->reweighted = false;
    struct EventList { /* an early error return destroys the events that finish_events() has not collected */
        std::vector<EventPair> v;
        ~EventList() {
            for (auto &e : v) {
                cudaEventDestroy(e.a);
                cudaEventDestroy(e.b);
            }
        }
    } eventList;
    std::vector<EventPair> &events = eventList.v;
    auto tic = [&](double *sink) {
        EventPair e;
        cudaEventCreate(&e.a);
        cudaEventCreate(&e.b);
        e.sink = sink;
        cudaEventRecord(e.a, st);
        events.push_back(e);
        return events.size() - 1;
    };
    auto toc = [&](size_t id) { cudaEventRecord(events[id].b, st); };
    auto finish_events = [&]() {
        for (auto &e : events) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) *e.sink += ms;
            cudaEventDestroy(e.a);
            cudaEventDestroy(e.b);
        }
        events.clear();
    };

    /* CPB_HOST_TIMING=1: wall-clock stamps (with a stream synchronisation each) at the stages of a run, on stderr */
    const bool hostTiming = getenv("CPB_HOST_TIMING") != nullptr;
    auto wall = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double tStamp = wall();
    auto stamp = [&](const char *what) {
        if (!hostTiming) return;
        cudaStreamSynchronize(st);
        const double now = wall();
        fprintf(stderr, "  [run] %-28s %9.3f ms\n", what, now - tStamp);
        tStamp = now;
    };

    const int nPlanes = mode == CPB_MODE_FORWARD ? 0 : (mode == CPB_MODE_ALIGNED_PAIRS ? 1 : (mode == CPB_MODE_ALIGNED_PAIRS_INDELS ? 3 : S));
    const int auxF = (mode == CPB_MODE_ALIGNED_PAIRS || mode == CPB_MODE_ALIGNED_PAIRS_INDELS) ? S : 0;
    const int nLists = mode == CPB_MODE_ALIGNED_PAIRS ? 1 : (mode == CPB_MODE_ALIGNED_PAIRS_INDELS ? 3 : 0);
    const int hmmLen = CPB_HMM_LEN(S);

    int rc = CPB_OK;
    for (int l = 0; l < 3; l++) {
        b->outCount[l] = 0;
        b->pairOff[l].assign(b->n + 1, 0);
    }
    b->lastMode = mode;
    b->lastS = S;
    if (mode == CPB_MODE_EXPECTATIONS) {
        if ((rc = b->perPair.reserve(std::max<int64_t>(b->n, 1) * hmmLen * sizeof(double))) != CPB_OK) return rc;
        if ((rc = b->hmmTotal.reserve(hmmLen * sizeof(double))) != CPB_OK) return rc;
        CUDA_TRY(cudaMemsetAsync(b->perPair.p, 0, std::max<int64_t>(b->n, 1) * hmmLen * sizeof(double), st));
        CUDA_TRY(cudaMemsetAsync(b->hmmTotal.p, 0, hmmLen * sizeof(double), st));
    }

    /* The plan of a run -- regions, bands, traceback schedule, chunks, work lists -- depends on the batch, the mode, the state count
     * and the banding parameters, not on the model's numbers: a batch that is run again with the same ones (every EM iteration of a
     * resident batch) keeps its plan, host tables and device tables alike.  $CPB_NO_PLAN_CACHE=1 plans every run anew. */
    HostArray<RegionDev> &regs = b->hRegions;
    HostArray<BlockRec> &hBlocks = b->hBlocks;
    std::vector<Chunk> &chunks = b->chunks;
    int64_t nReg = 0, nDiagRecs = 0, totalBlocks = 0;
    size_t scratchNeed = 0;
    PlanKey key;
    memset(&key, 0, sizeof(key));
    key.mode = mode;
    key.states = S;
    key.split = p->splitMatrixBiggerThanThis;
    key.expansion = p->diagonalExpansion;
    key.dynamic = p->dynamicAnchorExpansion != 0;
    key.minDiags = p->minDiagsBetweenTraceBack;
    key.traceBack = p->traceBackDiagonals;
    key.budget = (int64_t) ctx->scratchBudget;
    auto make_plan = [&]() -> int {
        int rc = CPB_OK;
        /* where the pairs are cut into regions: decided on the device, which has the anchors; the host gets one bit per gap */
        const uint32_t *hostFlags = nullptr;
        struct PinnedLoan { /* goes back to the context's pool when the plan is made, or on an error return */
            PinnedPool *pool = nullptr;
            void *p = nullptr;
            ~PinnedLoan() {
                if (p != nullptr) pool->give(p);
            }
        } loan;
        std::vector<uint32_t> pageable;
        if (mode != CPB_MODE_FORWARD && b->n > 0) {
            const int64_t nBits = b->aOff[b->n] + b->n;
            const size_t words = (size_t) ((nBits + 31) / 32 + 1), head = 4; /* word 0: pairs with a cut; the bits start at word 4 */
            if ((rc = b->splitFlags.reserve((head + words) * sizeof(uint32_t))) != CPB_OK) return rc;
            uint32_t *dFlags = b->splitFlags.as<uint32_t>();
            CUDA_TRY(cudaMemsetAsync(dFlags, 0, (head + words) * sizeof(uint32_t), st));
            const int64_t *tab = b->dPairTab.as<int64_t>();
            k_split_flags<<<(unsigned) ((b->n * 32 + 255) / 256), 256, 0, st>>>(b->dAnchors.as<int32_t>(), tab, tab + (b->n + 1), tab + 2 * (b->n + 1), (int) b->n,
                                                                              (long long) p->splitMatrixBiggerThanThis, dFlags + head, dFlags);
            stx.kernelLaunches++;
            uint32_t cutPairs = 0;
            CUDA_TRY(cudaMemcpyAsync(&cutPairs, dFlags, sizeof(cutPairs), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            CUDA_TRY(cudaGetLastError());
            if (cutPairs > 0) {
                loan.pool = &ctx->pinned;
                loan.p = ctx->pinned.take(words * sizeof(uint32_t));
                uint32_t *dst = static_cast<uint32_t *>(loan.p);
                if (dst == nullptr) {
                    pageable.resize(words);
                    dst = pageable.data();
                }
                CUDA_TRY(cudaMemcpyAsync(dst, dFlags + head, words * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaStreamSynchronize(st));
                hostFlags = dst;
            }
        }
        stamp("k_split_flags");
        rc = build_regions(b, p, mode, hostFlags);
        if (rc != CPB_OK) return rc;
        stamp("build_regions");
        nReg = (int64_t) regs.size();
        stx.nRegions = nReg;
        if (nReg == 0) return CPB_OK;
        nDiagRecs = regs.back().diagBase + regs.back().lX + regs.back().lY + 3;
        const int64_t blockSlots = regs.back().blockBase + regs.back().blockCap;
        stx.diagonals = nDiagRecs - 2 * nReg; /* lX+lY+1 per region */

        if ((rc = b->regions.reserve(nReg * sizeof(RegionDev))) != CPB_OK) return rc;
        if ((rc = b->diags.reserve(nDiagRecs * sizeof(DiagRec))) != CPB_OK) return rc;
        if ((rc = b->blocks.reserve(blockSlots * sizeof(BlockRec))) != CPB_OK) return rc;
        const int64_t nStripRecs = regs.back().stripBase + (regs.back().lX >> 5) + 1;
        if ((rc = b->strips.reserve(nStripRecs * sizeof(StripRec))) != CPB_OK) return rc;
        if (mode != CPB_MODE_FORWARD) {
            if ((rc = b->totals.reserve(nDiagRecs * sizeof(double))) != CPB_OK) return rc;
        } else {
            if ((rc = b->forwardOut.reserve(nReg * sizeof(double))) != CPB_OK) return rc;
        }
        CUDA_TRY(cudaMemcpyAsync(b->regions.p, regs.data(), nReg * sizeof(RegionDev), cudaMemcpyHostToDevice, st));

        /* K1: band + schedule */
        {
            BandArgs ba;
            ba.regions = b->regions.as<RegionDev>();
            ba.anchors = b->dAnchors.as<int32_t>();
            ba.diags = b->diags.as<DiagRec>();
            ba.blocks = b->blocks.as<BlockRec>();
            ba.strips = b->strips.as<StripRec>();
            ba.nRegions = (int32_t) nReg;
            ba.expansion = (int32_t) p->diagonalExpansion;
            ba.dynamic = (mode == CPB_MODE_FORWARD) ? 0 : (p->dynamicAnchorExpansion != 0); /* forward prob always uses the static band (:894) */
            ba.minDiags = (int32_t) p->minDiagsBetweenTraceBack;
            ba.traceBack = (int32_t) p->traceBackDiagonals;
            ba.auxF = auxF;
            ba.scheduleOn = mode != CPB_MODE_FORWARD;
            size_t ev = tic(&stx.msBand);
            k_band<<<(unsigned) ((nReg + BAND_WARPS - 1) / BAND_WARPS), 32 * BAND_WARPS, 0, st>>>(ba);
            toc(ev);
            stx.kernelLaunches++;
        }
        CUDA_TRY(cudaMemcpyAsync(regs.data(), b->regions.p, nReg * sizeof(RegionDev), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaGetLastError());

        stamp("k_band + region sizes");
        /* validate, gather the block table in compact region order */
        totalBlocks = 0;
        for (int64_t r = 0; r < nReg; r++) {
            if (regs[r].err == 1) {
                cpb_set_error("pair %d: anchors produce an invalid band diagonal (PAIRWISE_ALIGNMENT_EXCEPTION in the reference)", regs[r].pair);
                finish_events();
                return CPB_ERR_BAND;
            }
            if (regs[r].err == 2) {
                cpb_set_error("internal: traceback block table overflow for pair %d", regs[r].pair);
                finish_events();
                return CPB_ERR_BAND;
            }
            if (regs[r].cells >= ((int64_t) 1 << 31)) {
                cpb_set_error("pair %d: a single region has %lld band cells (limit 2^31)", regs[r].pair, (long long) regs[r].cells);
                finish_events();
                return CPB_ERR_ARGUMENT;
            }
            totalBlocks += regs[r].nBlocks;
            stx.cells += regs[r].cells;
            stx.maxWidth = std::max(stx.maxWidth, regs[r].maxW);
        }
        stx.nBlocks = totalBlocks;
        if (!hBlocks.resize((size_t) totalBlocks)) {
            cpb_set_error("out of host memory for %lld block records", (long long) totalBlocks);
            return CPB_ERR_MEMORY;
        }
        std::vector<int64_t> regionBlock0(nReg + 1, 0);
        if (totalBlocks > 0) {
            HostArray<BlockRec> slots; /* the slots as k_band filled them: blockCap per region, nBlocks of them used */
            slots.pool = &ctx->pinned;
            if (!slots.resize((size_t) blockSlots)) {
                cpb_set_error("out of host memory for %lld block slots", (long long) blockSlots);
                return CPB_ERR_MEMORY;
            }
            CUDA_TRY(cudaMemcpyAsync(slots.data(), b->blocks.p, blockSlots * sizeof(BlockRec), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            int64_t k = 0;
            for (int64_t r = 0; r < nReg; r++) {
                regionBlock0[r] = k;
                for (int j = 0; j < regs[r].nBlocks; j++) {
                    hBlocks[k] = slots[regs[r].blockBase + j];
                    hBlocks[k++].ckBase = -1;
                }
            }
            regionBlock0[nReg] = k;
            CUDA_TRY(cudaMemcpyAsync(b->blocks.p, hBlocks.data(), totalBlocks * sizeof(BlockRec), cudaMemcpyHostToDevice, st));
        }

        stamp("block table");
        /* chunk planning */
        const int64_t bytesPerCell = (int64_t) sizeof(double) * 2 * nPlanes;
        for (int attempt = 0;; attempt++) {
            bool budgetFromCache = false;
            size_t budget = ctx->scratchBudget;
            if (budget == 0) {
                /* 70 % of what is free; a run that fits the scratch buffer already there does not need to ask the driver (cudaMemGetInfo
                 * costs tens of milliseconds once a few hundred buffers are live) */
                size_t wholeRun = 0;
                for (int64_t r = 0; r < nReg; r++) wholeRun += (size_t) ((regs[r].cells + 36) * bytesPerCell + (regs[r].auxDoubles + 6) * 8);
                if (wholeRun + 256 <= ctx->scratch.cap) {
                    budget = ctx->scratch.cap;
                } else {
                    budgetFromCache = ctx->freeEpoch == g_allocEpoch.load();
                    if (!budgetFromCache) {
                        size_t freeB = 0, totalB = 0;
                        CUDA_TRY(cudaMemGetInfo(&freeB, &totalB));
                        ctx->freePlusScratch = freeB + ctx->scratch.cap;
                        ctx->freeEpoch = g_allocEpoch.load();
                    }
                    budget = (size_t) ((double) ctx->freePlusScratch * 0.70);
                }
            }
            chunks.clear();
            {
                int64_t r = 0;
                while (r < nReg) {
                    Chunk c;
                    memset(&c, 0, sizeof(c));
                    c.region0 = r;
                    int64_t cells = 0, aux = 0, words = 0;
                    while (r < nReg) {
                        const int64_t nc = cells + regs[r].cells + 32, na = aux + regs[r].auxDoubles + 4;
                        if (r > c.region0 && (size_t) (nc * bytesPerCell + na * 8) > budget) break;
                        regs[r].cellBase = cells;
                        regs[r].auxBase = aux;
                        regs[r].maskBase = words;
                        cells = (nc + 3) & ~int64_t(3);
                        aux = (na + 1) & ~int64_t(1);
                        words += (regs[r].cells >> 5) + regs[r].lX + regs[r].lY + 4;
                        r++;
                    }
                    c.region1 = r;
                    c.cells = cells;
                    c.aux = aux;
                    c.maskWords = words; /* provisional; final value below once the decades are counted */
                    c.stride = (cells + 31) & ~int64_t(31);
                    c.block0 = regionBlock0[c.region0];
                    c.block1 = regionBlock0[c.region1];
                    c.pair0 = regs[c.region0].pair;
                    c.pair1 = regs[c.region1 - 1].pair;
                    /* decades: ceil(owned diagonals / 10) per block, numbered consecutively inside the chunk */
                    int64_t dec = 0;
                    for (int64_t k = c.block0; k < c.block1; k++) {
                        hBlocks[k].decadeBase = dec;
                        dec += (hBlocks[k].from - hBlocks[k].T + 9) / 10;
                    }
                    c.decades = dec;
                    c.maskWords = (c.cells >> 5) + dec + 2; /* k_posterior: word of chunk cell C in decade g is (C >> 5) + g */
                    chunks.push_back(c);
                }
            }
            stx.nChunks = (int64_t) chunks.size();
            stamp("chunk planning");
            if (totalBlocks > 0) CUDA_TRY(cudaMemcpyAsync(b->blocks.p, hBlocks.data(), totalBlocks * sizeof(BlockRec), cudaMemcpyHostToDevice, st));
            scratchNeed = 0;
            for (auto &c : chunks) scratchNeed = std::max(scratchNeed, (size_t) (c.stride * bytesPerCell + c.aux * 8 + 256));
            rc = ctx->scratch.reserve(std::max<size_t>(scratchNeed, 256));
            if (rc == CPB_OK) break;
            /* the budget may rest on an answer of cudaMemGetInfo from before somebody else in this process took device memory: ask again, once */
            if (attempt > 0 || !budgetFromCache) return rc;
            (void) cudaGetLastError();
            ctx->freeEpoch = 0;

        }
        stamp("scratch");
        /* launch lists: forward regions per class, backward blocks per class, all blocks in order */
        std::vector<int32_t> lists;
        {
            int64_t total = 0;
            for (auto &c : chunks) {
                c.allBlocksOff = total;
                c.stripFwdOff = c.allBlocksOff + (c.block1 - c.block0);
                c.stripBwdOff = c.stripFwdOff + (c.region1 - c.region0);
                total = c.stripBwdOff + (c.block1 - c.block0);
            }
            lists.resize((size_t) total);
            /* strip engine: one list of regions and one of blocks per chunk, most expensive first (work is fetched dynamically); the
             * block lists are ordered by a second thread while this one does the regions */
            auto block_lists = [&]() {
                for (auto &c : chunks) {
                    int32_t *all = lists.data() + c.allBlocksOff, *bwd = lists.data() + c.stripBwdOff;
                    for (int64_t k = c.block0; k < c.block1; k++) all[k - c.block0] = bwd[k - c.block0] = (int32_t) k;
                    order_by_cost_descending(bwd, c.block1 - c.block0, [&](int32_t k) { return (int64_t) hBlocks[(size_t) k].cells; });
                }
            };
            auto region_lists = [&]() {
                for (auto &c : chunks) {
                    int32_t *fwd = lists.data() + c.stripFwdOff;
                    for (int64_t r = c.region0; r < c.region1; r++) fwd[r - c.region0] = (int32_t) r;
                    order_by_cost_descending(fwd, c.region1 - c.region0, [&](int32_t x) { return (int64_t) regs[(size_t) x].cells; });
                }
            };
            if (total > 100000) {
                std::thread other(block_lists);
                region_lists();
                other.join();
            } else {
                block_lists();
                region_lists();
            }
        }
        if ((rc = b->lists.reserve(std::max<size_t>(lists.size(), 1) * sizeof(int32_t))) != CPB_OK) return rc;
        CUDA_TRY(cudaMemcpyAsync(b->lists.p, lists.data(), lists.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(b->regions.p, regs.data(), nReg * sizeof(RegionDev), cudaMemcpyHostToDevice, st));

        stamp("lists");
        return CPB_OK;
    };
    bool reuse = b->planValid && memcmp(&key, &b->planKey, sizeof(key)) == 0 && getenv("CPB_NO_PLAN_CACHE") == nullptr;
    if (reuse && ctx->scratch.reserve(std::max<size_t>(b->planScratch, 256)) != CPB_OK) {
        /* the context's scratch has served another batch since and the chunks of the kept plan no longer fit what is free: plan anew */
        (void) cudaGetLastError();
        reuse = false;
    }
    if (reuse) {
        nReg = (int64_t) regs.size();
        nDiagRecs = regs.back().diagBase + regs.back().lX + regs.back().lY + 3;
        totalBlocks = (int64_t) hBlocks.size();
        scratchNeed = b->planScratch;
        stx.nRegions = b->planStats.nRegions;
        stx.diagonals = b->planStats.diagonals;
        stx.cells = b->planStats.cells;
        stx.maxWidth = b->planStats.maxWidth;
        stx.nBlocks = b->planStats.nBlocks;
        stx.nChunks = b->planStats.nChunks;
        stx.planReused = 1;
        stamp("plan reused");
    } else {
        b->planValid = false;
        if ((rc = make_plan()) != CPB_OK) return rc;
        if (nReg > 0) {
            b->planKey = key;
            b->planStats = stx;
            b->planScratch = scratchNeed;
            b->planValid = true;
        }
    }
    if (nReg == 0) {
        CUDA_TRY(cudaStreamSynchronize(st));
        return CPB_OK;
    }
    int64_t maxChunkBlocks = 1, maxDecades = 1, maxMaskWords = 1, maxChunkPairs = 1;
    for (auto &c : chunks) {
        maxChunkBlocks = std::max(maxChunkBlocks, c.block1 - c.block0);
        maxDecades = std::max(maxDecades, c.decades);
        maxMaskWords = std::max(maxMaskWords, c.maskWords);
        maxChunkPairs = std::max(maxChunkPairs, c.pair1 - c.pair0 + 1);
    }
    const int64_t maxTiles = (maxDecades + SCAN_TILE - 1) / SCAN_TILE;
    if (nLists > 0) {
        if ((rc = b->counts.reserve((size_t) nLists * maxDecades * sizeof(int32_t))) != CPB_OK) return rc;
        if ((rc = b->offsets.reserve((size_t) nLists * maxDecades * sizeof(int64_t))) != CPB_OK) return rc;
        if ((rc = b->masks.reserve((size_t) nLists * maxMaskWords * sizeof(uint32_t))) != CPB_OK) return rc;
        if ((rc = b->tileSums.reserve((size_t) (nLists * maxTiles + 8) * sizeof(int64_t))) != CPB_OK) return rc;
        if ((rc = b->pairCounts.reserve((size_t) nLists * std::max<int64_t>(b->n, 1) * sizeof(int64_t))) != CPB_OK) return rc;
        if ((rc = b->pairBlockOff.reserve((size_t) (maxChunkPairs + 2) * sizeof(int64_t))) != CPB_OK) return rc;
        CUDA_TRY(cudaMemsetAsync(b->pairCounts.p, 0, (size_t) nLists * std::max<int64_t>(b->n, 1) * sizeof(int64_t), st));
    }
    if (mode == CPB_MODE_EXPECTATIONS) {
        if ((rc = b->partials.reserve(maxChunkBlocks * hmmLen * sizeof(double))) != CPB_OK) return rc;
        if ((rc = b->pairBlockOff.reserve((size_t) (maxChunkPairs + 2) * sizeof(int64_t))) != CPB_OK) return rc;
    }

    stamp("planning + lists");
    /* strip engine: persistent grid of independent warps, boundary rings, work counters */
    typedef void (*StripKernel)(const DpArgs, const CpbModel, const StripArgs);
    StripKernel kFwdStrip = nullptr, kFwdTeam = nullptr, kFwdBlocks = nullptr, kBwdStrip = nullptr;
    /* the backward kernel exists compiled for 6 and for 3 resident CTAs per SM: see strip_kernels.cuh ($CPB_BWD_WIDE=0/1 forces one) */
    bool bwdWide = stx.maxWidth > kBwdWideBand;
    if (getenv("CPB_BWD_WIDE") != nullptr) bwdWide = atoi(getenv("CPB_BWD_WIDE")) != 0;
    StripKernel kCkStrip = k_forward_strip<S, 0, kStripWPC, FWD_REGIONS>, kCkTeam = k_forward_strip<S, 0, kStripWPC, FWD_TEAMS>; /* first pass of two */
    switch (mode) {
    case CPB_MODE_FORWARD:
        kFwdStrip = k_forward_strip<S, 0, kStripWPC, FWD_REGIONS>;
        kFwdTeam = k_forward_strip<S, 0, kStripWPC, FWD_TEAMS>;
        kBwdStrip = bwdWide ? k_backward_strip<S, 0, true, kStripWPC, CPB_BWD_WIDE_MIN_BLOCKS> : k_backward_strip<S, 0, true, kStripWPC, CPB_BWD_MIN_BLOCKS>;
        break;
    case CPB_MODE_ALIGNED_PAIRS:
        kFwdStrip = k_forward_strip<S, 1, kStripWPC, FWD_REGIONS>;
        kFwdTeam = k_forward_strip<S, 1, kStripWPC, FWD_TEAMS>;
        kFwdBlocks = k_forward_strip<S, 1, kStripWPC, FWD_BLOCKS>;
        kBwdStrip = bwdWide ? k_backward_strip<S, 1, true, kStripWPC, CPB_BWD_WIDE_MIN_BLOCKS> : k_backward_strip<S, 1, true, kStripWPC, CPB_BWD_MIN_BLOCKS>;
        break;
    case CPB_MODE_ALIGNED_PAIRS_INDELS:
        kFwdStrip = k_forward_strip<S, 3, kStripWPC, FWD_REGIONS>;
        kFwdTeam = k_forward_strip<S, 3, kStripWPC, FWD_TEAMS>;
        kFwdBlocks = k_forward_strip<S, 3, kStripWPC, FWD_BLOCKS>;
        kBwdStrip = bwdWide ? k_backward_strip<S, 3, true, kStripWPC, CPB_BWD_WIDE_MIN_BLOCKS> : k_backward_strip<S, 3, true, kStripWPC, CPB_BWD_MIN_BLOCKS>;
        break;
    default:
        kFwdStrip = k_forward_strip<S, S, kStripWPC, FWD_REGIONS>;
        kFwdTeam = k_forward_strip<S, S, kStripWPC, FWD_TEAMS>;
        kFwdBlocks = k_forward_strip<S, S, kStripWPC, FWD_BLOCKS>;
        kBwdStrip = bwdWide ? k_backward_strip<S, S, false, kStripWPC, CPB_BWD_WIDE_MIN_BLOCKS> : k_backward_strip<S, S, false, kStripWPC, CPB_BWD_MIN_BLOCKS>;
        break;
    }
    /* narrow bands: groups of 8 or 16 lanes per region / block (narrow_kernels.cuh) */
    typedef void (*NarrowKernel)(const DpArgs, const CpbModel, const NarrowArgs);
    auto narrow_forward = [&](int G) -> NarrowKernel {
        switch (mode) {
        case CPB_MODE_ALIGNED_PAIRS:
            return G == 8 ? k_forward_narrow<S, 1, 8, kStripWPC> : (G == 16 ? k_forward_narrow<S, 1, 16, kStripWPC> : k_forward_narrow<S, 1, 32, kStripWPC>);
        case CPB_MODE_ALIGNED_PAIRS_INDELS:
            return G == 8 ? k_forward_narrow<S, 3, 8, kStripWPC> : (G == 16 ? k_forward_narrow<S, 3, 16, kStripWPC> : k_forward_narrow<S, 3, 32, kStripWPC>);
        default:
            return G == 8 ? k_forward_narrow<S, S, 8, kStripWPC> : (G == 16 ? k_forward_narrow<S, S, 16, kStripWPC> : k_forward_narrow<S, S, 32, kStripWPC>);
        }
    };
    auto narrow_backward = [&](int G) -> NarrowKernel {
        switch (mode) {
        case CPB_MODE_ALIGNED_PAIRS:
            return G == 8 ? k_backward_narrow<S, 1, true, 8, kStripWPC>
                          : (G == 16 ? k_backward_narrow<S, 1, true, 16, kStripWPC> : k_backward_narrow<S, 1, true, 32, kStripWPC>);
        case CPB_MODE_ALIGNED_PAIRS_INDELS:
            return G == 8 ? k_backward_narrow<S, 3, true, 8, kStripWPC>
                          : (G == 16 ? k_backward_narrow<S, 3, true, 16, kStripWPC> : k_backward_narrow<S, 3, true, 32, kStripWPC>);
        default:
            return G == 8 ? k_backward_narrow<S, S, false, 8, kStripWPC>
                          : (G == 16 ? k_backward_narrow<S, S, false, 16, kStripWPC> : k_backward_narrow<S, S, false, 32, kStripWPC>);
        }
    };
    StripArgs sargs;
    memset(&sargs, 0, sizeof(sargs));
    int stripGrid = 1, teamGrid = 1, fwdGrid = 1, bwdGrid = 1; /* stripGrid = the larger of the two: sizes the rings */
    {
        int maxRange = 1;
        for (int64_t r = 0; r < nReg; r++) maxRange = std::max(maxRange, regs[r].maxStripRange);
        int ring = 64;
        while (ring < maxRange + 4) ring <<= 1;
        int occF = 1, occB = 1, occT = 1;
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occF, kFwdStrip, 32 * kStripWPC, 0));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occB, kBwdStrip, 32 * kStripWPC, 0));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occT, kFwdTeam, 32 * kStripWPC, 0));
        fwdGrid = ctx->smCount * std::max(1, occF);
        bwdGrid = ctx->smCount * std::max(1, occB);
        stripGrid = std::max(fwdGrid, bwdGrid);
        teamGrid = ctx->smCount * std::max(1, std::min(occT, occF)); /* every team CTA must be resident: teams spin on each other */
        if ((rc = ctx->progress.reserve((size_t) stripGrid * kStripWPC * sizeof(unsigned long long))) != CPB_OK) return rc;
        sargs.progress = ctx->progress.as<unsigned long long>();
        const size_t need = (size_t) stripGrid * kStripWPC * 2 * ring * BND_REC * sizeof(double);
        if ((rc = ctx->boundary.reserve(need)) != CPB_OK) return rc;
        if ((rc = ctx->counters.reserve(2 * chunks.size() * sizeof(unsigned int) + 16)) != CPB_OK) return rc;
        CUDA_TRY(cudaMemsetAsync(ctx->counters.p, 0, 2 * chunks.size() * sizeof(unsigned int) + 16, st));
        sargs.strips = b->strips.as<StripRec>();
        sargs.boundary = ctx->boundary.as<double>();
        sargs.negRecord = ctx->negRecord.as<double>();
        sargs.ringSize = ring;
    }

    /* How many warps of a team share one region when `cnt` regions of `cells` cells in all are launched together: the largest
     * power of two that still keeps every warp slot busy, at most 16 (a strip lags its predecessor by ~64 diagonals); 1 for short
     * regions, where a hand-over between warps costs more than a strip. */
    auto team_size = [&](int64_t cnt, int64_t cells) {
        int team = 1;
        if (cnt > 0 && cells / cnt >= (int64_t) 1 << 20) {
            while (team < 16 && cnt * team * 2 <= (int64_t) teamGrid * kStripWPC) team *= 2;
        }
        if (getenv("CPB_TEAM") != nullptr) team = std::max(1, atoi(getenv("CPB_TEAM")));
        return team;
    };
    auto launch_forward_regions = [&](StripKernel plain, StripKernel teamed, const DpArgs &a, int64_t cnt, int64_t cells) {
        const int team = team_size(cnt, cells);
        if (team > 1 || getenv("CPB_TEAM_KERNEL") != nullptr) {
            const int grid = (int) std::min<int64_t>(teamGrid, (cnt * team + kStripWPC - 1) / kStripWPC);
            sargs.teamSize = team;
            cudaMemsetAsync(ctx->progress.p, 0, (size_t) grid * kStripWPC * sizeof(unsigned long long), st);
            teamed<<<grid, 32 * kStripWPC, 0, st>>>(a, *m, sargs);
        } else {
            const int grid = (int) std::min<int64_t>(fwdGrid, (cnt + kStripWPC - 1) / kStripWPC);
            sargs.teamSize = 1;
            plain<<<grid, 32 * kStripWPC, 0, st>>>(a, *m, sargs);
        }
        stx.kernelLaunches++;
#ifdef CPB_TEAM_DEBUG
        if (team > 1) {
            unsigned long long dbg[8] = { 0 }, zero[8] = { 0 };
            cudaStreamSynchronize(st);
            cudaMemcpyFromSymbol(dbg, g_teamDebug, sizeof(dbg));
            cudaMemcpyToSymbol(g_teamDebug, zero, sizeof(zero));
            fprintf(stderr, "team %d, %lld regions: %llu wait calls, %llu spun, %llu spin iterations, %.3f ms waiting; %llu publishes, %.3f ms publishing (summed over warps)\n",
                    team, (long long) cnt, dbg[3], dbg[1], dbg[2], (double) dbg[0] / 1.965e6, dbg[5], (double) dbg[4] / 1.965e6);
        }
#endif
        return team;
    };

    /*
     * Two-pass forward.  A chunk of few, long regions (one whose forward sweep would need teams) leaves most of the machine idle: a
     * region is one sequential sweep and a team only gets as many warps going as the band is wide.  Such runs instead make one
     * plane-less sweep over ALL regions of the batch at once (no HBM planes, so no chunking: every region is in flight), keeping
     * the full cells of the two diagonals in front of every traceback block; then, chunk by chunk, every block recomputes its own
     * forward cells from its checkpoint -- as many work items as blocks.  Same arithmetic in the same order: bit-identical planes.
     */
    bool twoPass = false;
    if (mode != CPB_MODE_FORWARD && totalBlocks > nReg) {
        /* it pays when chunking is what starves the machine: the first pass then has several chunks' worth of regions in flight */
        for (auto &c : chunks) {
            int64_t cells = 0;
            for (int64_t r = c.region0; r < c.region1; r++) cells += regs[r].cells;
            if (chunks.size() > 1 && team_size(c.region1 - c.region0, cells) > 1) twoPass = true;
        }
        if (getenv("CPB_TWO_PASS") != nullptr) twoPass = atoi(getenv("CPB_TWO_PASS")) != 0;
        for (int64_t k = 0; k < totalBlocks && twoPass; k++) {
            /* diagonal 0 is not stored through the aux path, and the checkpoint diagonals of two blocks must not coincide
             * (library defaults put block starts >= 960 diagonals apart) */
            if (hBlocks[k].T == 1) twoPass = false;
            if (k > 0 && hBlocks[k].region == hBlocks[k - 1].region && hBlocks[k].T - hBlocks[k - 1].T < 2) twoPass = false;
        }
    }
    if (twoPass) {
        std::vector<int32_t> sizes(totalBlocks);
        if ((rc = b->ckSizes.reserve(totalBlocks * sizeof(int32_t))) != CPB_OK) return rc;
        k_ckpt_sizes<<<(unsigned) ((totalBlocks + 255) / 256), 256, 0, st>>>(b->blocks.as<BlockRec>(), b->regions.as<RegionDev>(), b->diags.as<DiagRec>(),
                                                                         (int) totalBlocks, S, b->ckSizes.as<int32_t>());
        CUDA_TRY(cudaMemcpyAsync(sizes.data(), b->ckSizes.p, totalBlocks * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        int64_t total = 0;
        for (int64_t k = 0; k < totalBlocks; k++) {
            hBlocks[k].ckBase = total;
            total += sizes[k];
        }
        if (total >= ((int64_t) 1 << 32)) {
            twoPass = false; /* aux offsets are 32-bit */
        } else {
            CUDA_TRY(cudaMemcpyAsync(b->blocks.p, hBlocks.data(), totalBlocks * sizeof(BlockRec), cudaMemcpyHostToDevice, st));
            if ((rc = b->ckpt.reserve(std::max<int64_t>(total, 1) * sizeof(double))) != CPB_OK) return rc;
            if ((rc = b->ckDiags.reserve(nDiagRecs * sizeof(DiagRec))) != CPB_OK) return rc;
            if ((rc = b->ckRegions.reserve(nReg * sizeof(RegionDev))) != CPB_OK) return rc;
            std::vector<RegionDev> ckRegs(regs.begin(), regs.end());
            for (auto &r : ckRegs) r.auxBase = 0; /* checkpoint offsets are absolute */
            CUDA_TRY(cudaMemcpyAsync(b->ckRegions.p, ckRegs.data(), nReg * sizeof(RegionDev), cudaMemcpyHostToDevice, st));
            k_ckpt_diags<<<(unsigned) ((nDiagRecs + 255) / 256), 256, 0, st>>>(b->diags.as<DiagRec>(), b->ckDiags.as<DiagRec>(), nDiagRecs);
            k_ckpt_mark<<<(unsigned) ((totalBlocks + 255) / 256), 256, 0, st>>>(b->blocks.as<BlockRec>(), b->regions.as<RegionDev>(), b->ckDiags.as<DiagRec>(),
                                                                            (int) totalBlocks, S);
            stx.kernelLaunches += 3;
            /* all regions, most expensive first */
            std::vector<int32_t> order(nReg);
            for (int64_t r = 0; r < nReg; r++) order[r] = (int32_t) r;
            order_by_cost_descending(order.data(), nReg, [&](int32_t x) { return (int64_t) regs[x].cells; });
            if ((rc = b->ckSizes.reserve(std::max<size_t>(totalBlocks * sizeof(int32_t), nReg * sizeof(int32_t)))) != CPB_OK) return rc;
            CUDA_TRY(cudaMemcpyAsync(b->ckSizes.p, order.data(), nReg * sizeof(int32_t), cudaMemcpyHostToDevice, st));
            DpArgs a1;
            memset(&a1, 0, sizeof(a1));
            a1.regions = b->ckRegions.as<RegionDev>();
            a1.blocks = b->blocks.as<BlockRec>();
            a1.diags = b->ckDiags.as<DiagRec>();
            a1.symX = b->symX.as<uint8_t>() + kSymPad;
            a1.symY = b->symY.as<uint8_t>() + kSymPad;
            a1.aux = b->ckpt.as<double>();
            a1.auxF = S;
            a1.list = b->ckSizes.as<int32_t>();
            sargs.counter = ctx->counters.as<unsigned int>() + 2 * chunks.size();
            sargs.nItems = (int32_t) nReg;
            size_t ev = tic(&stx.msCheckpoint);
            launch_forward_regions(kCkStrip, kCkTeam, a1, nReg, stx.cells);
            CUDA_TRY(cudaGetLastError());
            toc(ev);
            stx.twoPass = 1;
            CUDA_TRY(cudaStreamSynchronize(st)); /* `order` and `ckRegs` are read by the copies above */
        }
    }

    /* posterior scan: the keep threshold in log space under the host's libm, and the buffer for weights the host has to recompute */
    const double logThreshold = nLists > 0 ? log_threshold_for_host_libm(p->threshold) : 0.0;
    const double pintTolerance = getenv("CPB_PINT_TOLERANCE") != nullptr ? atof(getenv("CPB_PINT_TOLERANCE")) : 2e-8; /* tests: 0.5 sends every weight to the host */
    const int fixupCap = getenv("CPB_PINT_FIXUP_CAP") != nullptr ? atoi(getenv("CPB_PINT_FIXUP_CAP")) : 4096;
    if (nLists > 0) {
        if ((rc = ctx->fixups.reserve(16 + (size_t) fixupCap * sizeof(PintFixup))) != CPB_OK) return rc;
        CUDA_TRY(cudaMemsetAsync(ctx->fixups.p, 0, 16, st));
    }
    stamp("strip setup (+ checkpoint pass)");
    std::vector<int64_t> hPairOff;
    int64_t running[3] = { 0, 0, 0 }, sinkFrom[3] = { 0, 0, 0 };
    for (int l = 0; l < 3; l++) b->sunk[l] = l < nLists && b->sink[l] != nullptr;
    if (nLists > 0 && (b->sink[0] != nullptr || b->sink[1] != nullptr || b->sink[2] != nullptr) && ctx->copyStream == nullptr)
        CUDA_TRY(cudaStreamCreateWithFlags(&ctx->copyStream, cudaStreamNonBlocking));
    int64_t chunkIndex = -1;

    int64_t totalChunkCells = 0, cellsDone = 0;
    for (auto &c : chunks) totalChunkCells += c.cells;
    for (auto &c : chunks) {
        cellsDone += c.cells;
        DpArgs a;
        memset(&a, 0, sizeof(a));
        a.regions = b->regions.as<RegionDev>();
        a.blocks = b->blocks.as<BlockRec>();
        a.diags = b->diags.as<DiagRec>();
        a.symX = b->symX.as<uint8_t>() + kSymPad;
        a.symY = b->symY.as<uint8_t>() + kSymPad;
        double *scr = ctx->scratch.as<double>();
        a.planesF = scr;
        a.planesB = scr + (int64_t) nPlanes * c.stride;
        a.aux = scr + (int64_t) 2 * nPlanes * c.stride;
        a.totals = b->totals.as<double>();
        a.planeStride = c.stride;
        a.nPlanes = nPlanes;
        a.auxF = auxF;
        a.forwardOut = mode == CPB_MODE_FORWARD ? b->forwardOut.as<double>() : nullptr;
        const int32_t *dLists = b->lists.as<int32_t>();

        chunkIndex++;
        size_t ev = tic(&stx.msForward);
        /* narrow chunk: no diagonal of any of its regions has more than 32 cells */
        int narrowG = 0;
        if (mode != CPB_MODE_FORWARD && !twoPass) {
            int widest = 0;
            for (int64_t r = c.region0; r < c.region1; r++) widest = std::max(widest, regs[r].maxW);
            if (widest <= 32) narrowG = widest <= 8 ? 8 : (widest <= 16 ? 16 : 32);
            if (getenv("CPB_NARROW") != nullptr && atoi(getenv("CPB_NARROW")) == 0) narrowG = 0;
        }
        NarrowArgs nargs;
        memset(&nargs, 0, sizeof(nargs));
        auto launch_narrow = [&](NarrowKernel k, int64_t cnt) {
            const int64_t perCta = (int64_t) kStripWPC * (32 / narrowG);
            const int grid = (int) std::max<int64_t>(1, std::min<int64_t>(stripGrid, (cnt + perCta - 1) / perCta));
            nargs.nItems = (int32_t) cnt;
            k<<<grid, 32 * kStripWPC, 0, st>>>(a, *m, nargs);
            stx.kernelLaunches++;
        };
        if (narrowG != 0) {
            a.list = dLists + c.stripFwdOff;
            nargs.counter = ctx->counters.as<unsigned int>() + 2 * chunkIndex;
            launch_narrow(narrow_forward(narrowG), c.region1 - c.region0);
        } else if (twoPass) {
            /* every block of the chunk recomputes its forward cells from its checkpoint */
            const int64_t nbF = c.block1 - c.block0;
            a.ckpt = b->ckpt.as<double>();
            a.list = dLists + c.stripBwdOff;
            sargs.counter = ctx->counters.as<unsigned int>() + 2 * chunkIndex;
            sargs.nItems = (int32_t) nbF;
            sargs.teamSize = 1;
            const int grid = (int) std::min<int64_t>(fwdGrid, (nbF + kStripWPC - 1) / kStripWPC);
            kFwdBlocks<<<std::max(grid, 1), 32 * kStripWPC, 0, st>>>(a, *m, sargs);
            stx.kernelLaunches++;
        } else {
            const int64_t cnt = c.region1 - c.region0;
            a.list = dLists + c.stripFwdOff;
            sargs.counter = ctx->counters.as<unsigned int>() + 2 * chunkIndex;
            sargs.nItems = (int32_t) cnt;
            int64_t chunkCells = 0;
            for (int64_t r = c.region0; r < c.region1; r++) chunkCells += regs[r].cells;
            const int team = launch_forward_regions(kFwdStrip, kFwdTeam, a, cnt, chunkCells);
            (void) team;
        }
        toc(ev);
        if (mode == CPB_MODE_FORWARD) continue;

        const int64_t nb = c.block1 - c.block0;
        if (nb == 0) continue;
        ev = tic(&stx.msBackward);
        if (narrowG != 0) {
            a.list = dLists + c.stripBwdOff;
            nargs.counter = ctx->counters.as<unsigned int>() + 2 * chunkIndex + 1;
            launch_narrow(narrow_backward(narrowG), nb);
        } else {
            a.list = dLists + c.stripBwdOff;
            sargs.counter = ctx->counters.as<unsigned int>() + 2 * chunkIndex + 1;
            sargs.nItems = (int32_t) nb;
            const int grid = (int) std::min<int64_t>(bwdGrid, (nb + kStripWPC - 1) / kStripWPC);
            kBwdStrip<<<grid, 32 * kStripWPC, 0, st>>>(a, *m, sargs);
            stx.kernelLaunches++;
        }
        toc(ev);

        a.list = dLists + c.allBlocksOff;
        ev = tic(&stx.msTotals);
        k_totals<<<(unsigned) ((nb * 32 + 127) / 128), 128, 0, st>>>(a, (int) nb);
        stx.kernelLaunches++;
        toc(ev);

        /* decades of each pair are contiguous in the chunk: [pairDecade0[q], pairDecade0[q+1]) */
        const int64_t np = c.pair1 - c.pair0 + 1;
        if (nLists > 0) {
            PostArgs pa;
            memset(&pa, 0, sizeof(pa));
            pa.logThreshold = logThreshold;
            pa.pintTolerance = pintTolerance;
            pa.fixupCap = fixupCap;
            pa.fixupCount = ctx->fixups.as<unsigned int>();
            pa.fixups = reinterpret_cast<PintFixup *>(ctx->fixups.as<char>() + 16);
            pa.nLists = nLists;
            pa.nDecades = c.decades;
            pa.maskWords = c.maskWords;
            pa.counts = b->counts.as<int32_t>();
            pa.offsets = b->offsets.as<int64_t>();
            pa.masks = b->masks.as<uint32_t>();
            ev = tic(&stx.msPosterior);
            k_posterior<false><<<(unsigned) nb, 32 * POST_WARPS, 0, st>>>(a, pa);
            stx.kernelLaunches++;
            const int64_t nTiles = (c.decades + SCAN_TILE - 1) / SCAN_TILE;
            int64_t *tileSums = b->tileSums.as<int64_t>();
            int64_t *totalsOut = tileSums + (int64_t) nLists * maxTiles;
            for (int l = 0; l < nLists; l++) {
                const int32_t *cnt = pa.counts + (int64_t) l * c.decades;
                k_scan_tiles<<<(unsigned) nTiles, 256, 0, st>>>(cnt, c.decades, tileSums + l * maxTiles);
                k_scan_sums<<<1, 1, 0, st>>>(tileSums + l * maxTiles, nTiles, running[l], totalsOut + l);
                k_scan_apply<<<(unsigned) nTiles, 256, 0, st>>>(cnt, c.decades, tileSums + l * maxTiles, b->offsets.as<int64_t>() + (int64_t) l * c.decades);
                stx.kernelLaunches += 3;
            }
            hPairOff.assign(np + 1, 0);
            for (int64_t k = c.block0; k < c.block1; k++)
                hPairOff[regs[hBlocks[k].region].pair - c.pair0 + 1] += (hBlocks[k].from - hBlocks[k].T + 9) / 10;
            for (int64_t q = 0; q < np; q++) hPairOff[q + 1] += hPairOff[q];
            CUDA_TRY(cudaMemcpyAsync(b->pairBlockOff.p, hPairOff.data(), (np + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
            k_pair_counts<<<(unsigned) ((np * nLists + 127) / 128), 128, 0, st>>>(pa.counts, c.decades, nLists, b->pairBlockOff.as<int64_t>(), (int) np,
                                                                                  b->pairCounts.as<int64_t>() + c.pair0, std::max<int64_t>(b->n, 1));
            stx.kernelLaunches++;
            toc(ev);
            int64_t newTotals[3] = { 0, 0, 0 };
            CUDA_TRY(cudaMemcpyAsync(newTotals, totalsOut, nLists * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st)); /* also protects hPairOff */
            for (int l = 0; l < nLists; l++) {
                const size_t need = (size_t) std::max<int64_t>(newTotals[l], 1) * 3 * sizeof(int32_t);
                if (need > b->out[l].cap) {
                    /* grow, keeping what earlier chunks wrote */
                    /* size for the whole batch, extrapolating the yield of the chunks done so far */
                    DevBuf bigger;
                    bigger.pool = b->out[l].pool;
                    const double scale = 1.15 * (double) std::max<int64_t>(totalChunkCells, 1) / (double) std::max<int64_t>(cellsDone, 1);
                    if ((rc = bigger.reserve(std::max((size_t) ((double) need * std::max(scale, 1.0)), (size_t) 1 << 20))) != CPB_OK) return rc;
                    if (b->out[l].p && running[l] > 0)
                        CUDA_TRY(cudaMemcpyAsync(bigger.p, b->out[l].p, (size_t) running[l] * 3 * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
                    CUDA_TRY(cudaStreamSynchronize(st));
                    if (ctx->copyStream != nullptr) CUDA_TRY(cudaStreamSynchronize(ctx->copyStream)); /* copies out of the old buffer */
                    b->out[l].release();
                    b->out[l].adopt(bigger);
                }
                pa.out[l] = b->out[l].as<int32_t>();
                sinkFrom[l] = running[l];
                running[l] = newTotals[l];
            }
            ev = tic(&stx.msPosterior);
            k_posterior<true><<<(unsigned) nb, 32 * POST_WARPS, 0, st>>>(a, pa);
            stx.kernelLaunches++;
            toc(ev);
            /* result sinks: this chunk's triples go to the host on the copy stream while the next chunk's kernels run */
            for (int l = 0; l < nLists; l++) {
                if (b->sink[l] == nullptr || !b->sunk[l]) continue;
                if (running[l] > b->sinkCap[l]) {
                    b->sunk[l] = false; /* too small: cpb_batch_fetch_pairs will copy the list the ordinary way */
                    continue;
                }
                if (running[l] == sinkFrom[l]) continue;
                cudaEvent_t done;
                CUDA_TRY(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
                CUDA_TRY(cudaEventRecord(done, st));
                CUDA_TRY(cudaStreamWaitEvent(ctx->copyStream, done, 0));
                CUDA_TRY(cudaEventDestroy(done));
                CUDA_TRY(cudaMemcpyAsync(b->sink[l] + 3 * sinkFrom[l], b->out[l].as<int32_t>() + 3 * sinkFrom[l], (size_t) (running[l] - sinkFrom[l]) * 3 * sizeof(int32_t),
                                         cudaMemcpyDeviceToHost, ctx->copyStream));
            }
        } else if (mode == CPB_MODE_EXPECTATIONS) {
            const size_t smem = ((sizeof(Tables<S>) + 15) & ~size_t(15)) + (size_t) S * 16 * EXPECT_COLS * sizeof(double);
            ev = tic(&stx.msPosterior);
            k_expect<S><<<(unsigned) nb, 32, smem, st>>>(a, *m, b->partials.as<double>());
            stx.kernelLaunches++;
            hPairOff.assign(np + 1, 0);
            for (int64_t k = 0; k < nb; k++) hPairOff[regs[hBlocks[c.block0 + k].region].pair - c.pair0 + 1]++;
            for (int64_t q = 0; q < np; q++) hPairOff[q + 1] += hPairOff[q];
            CUDA_TRY(cudaMemcpyAsync(b->pairBlockOff.p, hPairOff.data(), (np + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
            k_reduce_pairs<<<(unsigned) ((np * hmmLen + 127) / 128), 128, 0, st>>>(b->partials.as<double>(), b->pairBlockOff.as<int64_t>(),
                                                                                    (int) np, hmmLen, b->perPair.as<double>() + c.pair0 * hmmLen);
            stx.kernelLaunches++;
            toc(ev);
            CUDA_TRY(cudaStreamSynchronize(st)); /* hPairOff is reused */
        }
    }
    if (mode == CPB_MODE_EXPECTATIONS) {
        size_t ev = tic(&stx.msPosterior);
        k_reduce_total<<<(unsigned) hmmLen, 256, 0, st>>>(b->perPair.as<double>(), (int) b->n, hmmLen, b->hmmTotal.as<double>());
        stx.kernelLaunches++;
        toc(ev);
    }
    std::vector<int64_t> hPairCounts;
    if (nLists > 0 && b->n > 0) {
        hPairCounts.resize((size_t) nLists * b->n);
        CUDA_TRY(cudaMemcpyAsync(hPairCounts.data(), b->pairCounts.p, hPairCounts.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
#ifdef CPB_LA_STATS
    {
        unsigned long long ls[4] = { 0, 0, 0, 0 }, zero[4] = { 0, 0, 0, 0 };
        cudaMemcpyFromSymbol(ls, g_laStats, sizeof(ls));
        cudaMemcpyToSymbol(g_laStats, zero, sizeof(zero));
        fprintf(stderr, "logAdd: %llu warp calls, %.1f%% with every lane beyond the cut-off; %llu lane calls, %.1f%% beyond the cut-off\n", ls[0],
                100.0 * ls[1] / (ls[0] ? ls[0] : 1), ls[2], 100.0 * ls[3] / (ls[2] ? ls[2] : 1));
    }
#endif
    stamp("chunks");
    if (nLists > 0) {
        /* Weights floor(p * 1e7) that sit within pintTolerance of an integer -- a few per 1e8 kept cells -- are recomputed here with the
         * host's libm, the function the reference itself calls (impl/pairwiseAligner.c:657-661), and patched into the device lists: the
         * triples are then identical to the reference's, not just equal up to the last place of exp. */
        unsigned int nFix = 0;
        CUDA_TRY(cudaMemcpyAsync(&nFix, ctx->fixups.p, sizeof(nFix), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (nFix > (unsigned) fixupCap) {
            cpb_set_error("posterior scan: %u weights need the host's exp, more than the fix-up buffer holds (%d); raise CPB_PINT_FIXUP_CAP", nFix, fixupCap);
            return CPB_ERR_MEMORY;
        }
        if (nFix > 0) {
            std::vector<PintFixup> fx(nFix);
            std::vector<int32_t> weights(nFix);
            CUDA_TRY(cudaMemcpyAsync(fx.data(), ctx->fixups.as<char>() + 16, nFix * sizeof(PintFixup), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            if (ctx->copyStream != nullptr) CUDA_TRY(cudaStreamSynchronize(ctx->copyStream)); /* the sinks are complete before they are patched */
            for (unsigned k = 0; k < nFix; k++) {
                double pr = exp(fx[k].lp);
                if (pr > 1.0) pr = 1.0;
                weights[k] = (int32_t) (int64_t) floor(pr * (double) CPB_PAIR_ALIGNMENT_PROB_1);
                CUDA_TRY(cudaMemcpyAsync(b->out[fx[k].list].as<int32_t>() + 3 * fx[k].pos, &weights[k], sizeof(int32_t), cudaMemcpyHostToDevice, st));
                if (b->sunk[fx[k].list]) b->sink[fx[k].list][3 * fx[k].pos] = weights[k];
            }
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        if (ctx->copyStream != nullptr) CUDA_TRY(cudaStreamSynchronize(ctx->copyStream));
        stx.pintFixups = nFix;
    }
    finish_events();
    stx.msForward += stx.msCheckpoint; /* the forward phase is both passes */
    for (int l = 0; l < nLists; l++) {
        b->outCount[l] = running[l];
        stx.outputTriples += running[l];
        for (int64_t i = 0; i < b->n; i++) b->pairOff[l][i + 1] = b->pairOff[l][i] + hPairCounts[(size_t) l * b->n + i];
    }
    return CPB_OK;
}

extern "C" int cpb_batch_run(cpb_batch *b, const CpbModel *m, const CpbParams *p, int mode) {
    if (b == nullptr || m == nullptr || p == nullptr || mode < CPB_MODE_ALIGNED_PAIRS || mode > CPB_MODE_FORWARD) {
        cpb_set_error("cpb_batch_run: bad argument");
        return CPB_ERR_ARGUMENT;
    }
    b->alnValid = false; /* the alignment list belongs to the lists of the run before */
    int rc = check_params(p);
    if (rc != CPB_OK) return rc;
    if (p->dynamicAnchorExpansion && mode != CPB_MODE_FORWARD && b->oddExpansionPair >= 0) {
        cpb_set_error("pair %lld: with dynamicAnchorExpansion every anchor's expansion must be even (impl/pairwiseAligner.c:166)",
                      (long long) b->oddExpansionPair);
        return CPB_ERR_ARGUMENT;
    }
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    if (m->stateNumber == 5) return run_impl<5>(b, m, p, mode);
    if (m->stateNumber == 3) return run_impl<3>(b, m, p, mode);
    cpb_set_error("cpb_batch_run: model has %d states (3 or 5 supported)", m->stateNumber);
    return CPB_ERR_ARGUMENT;
}

extern "C" int cpb_batch_set_result_sink(cpb_batch *b, int list, int32_t *hostTriples, int64_t capacityTriples) {
    if (b == nullptr || list < 0 || list > 2 || capacityTriples < 0) {
        cpb_set_error("cpb_batch_set_result_sink: bad argument");
        return CPB_ERR_ARGUMENT;
    }
    b->sink[list] = capacityTriples > 0 ? hostTriples : nullptr;
    b->sinkCap[list] = b->sink[list] != nullptr ? capacityTriples : 0;
    b->sunk[list] = false;
    return CPB_OK;
}

extern "C" void cpb_batch_stats(const cpb_batch *b, CpbRunStats *out) {
    if (b && out) *out = b->stats;
}

extern "C" int64_t cpb_batch_result_count(const cpb_batch *b, int list) {
    if (b == nullptr || list < 0 || list > 2) return 0;
    return b->outCount[list];
}

extern "C" const int32_t *cpb_batch_device_triples(const cpb_batch *b, int list) {
    if (b == nullptr || list < 0 || list > 2) return nullptr;
    return b->out[list].as<int32_t>();
}

extern "C" int cpb_batch_fetch_pairs(cpb_batch *b, int list, int64_t *offsets, int32_t *triples) {
    if (b == nullptr || list < 0 || list > 2 || (b->lastMode != CPB_MODE_ALIGNED_PAIRS && b->lastMode != CPB_MODE_ALIGNED_PAIRS_INDELS)) {
        cpb_set_error("cpb_batch_fetch_pairs: no aligned-pair results in this batch");
        return CPB_ERR_ARGUMENT;
    }
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    if (offsets) memcpy(offsets, b->pairOff[list].data(), (b->n + 1) * sizeof(int64_t));
    if (triples != nullptr && triples == b->sink[list] && b->sunk[list]) return CPB_OK; /* the run already delivered them there */
    if (triples && b->outCount[list] > 0) {
        CUDA_TRY(cudaMemcpyAsync(triples, b->out[list].p, (size_t) b->outCount[list] * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, b->ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(b->ctx->stream));
    }
    return CPB_OK;
}

/* The reference hands its lists back in the order its traceback produced them, reversed per region (impl/pairwiseAligner.c:1411-1418 pops
 * the region's list): regions ascending; inside a region the traceback blocks from last to first; inside a block the diagonals
 * ascending; along a diagonal x descending.  Order-sensitive callers (getMaximalExpectedAccuracyPairwiseAlignment walks the list
 * backwards and stops early) see the same list from us.  The device output is sorted by (x + y, x) per pair, and regions and blocks own
 * consecutive ranges of x + y, so this is a permutation of consecutive runs done on the host after the copy. */
extern "C" int cpb_batch_fetch_pairs_reference_order(cpb_batch *b, int list, int64_t *offsets, int32_t *triples) {
    const int rc = cpb_batch_fetch_pairs(b, list, offsets, triples);
    if (rc != CPB_OK || triples == nullptr) return rc;
    const std::vector<int64_t> &off = b->pairOff[list];
    const size_t nRegions = b->hRegions.size();
    if (nRegions == 0) return CPB_OK;
    /* position of every region's first block in the compact block order */
    std::vector<int64_t> firstBlock(nRegions + 1, 0);
    for (size_t r = 0; r < nRegions; r++) firstBlock[r + 1] = firstBlock[r] + b->hRegions[r].nBlocks;
    /* regions [r0, r1): r0 starts a pair and r1 ends one, so that every thread owns whole pairs */
    auto reorder = [&](size_t r0, size_t r1) {
        std::vector<int32_t> tmp;
        std::vector<std::pair<int64_t, int64_t>> runs; /* [first, last) triple of every block of the region */
        int64_t cur = 0;                               /* regions come in pair order and own ascending ranges of x + y: one sweep */
        int32_t pair = -1;
        for (size_t r = r0; r < r1; r++) {
            const RegionDev &R = b->hRegions[r];
            const int64_t pairEnd = off[R.pair + 1];
            if (R.pair != pair) {
                pair = R.pair;
                cur = off[pair];
            }
            const int64_t shift = (int64_t) R.ox + R.oy - 2; /* matrix diagonal d holds the sequence coordinates with x + y = d + shift */
            runs.clear();
            const int64_t regionFirst = cur;
            for (int j = 0; j < R.nBlocks; j++) {
                const int64_t hi = (int64_t) b->hBlocks[firstBlock[r] + j].from + shift;
                const int64_t first = cur;
                while (cur < pairEnd && (int64_t) triples[3 * cur + 1] + triples[3 * cur + 2] <= hi) cur++;
                runs.emplace_back(first, cur);
            }
            if (cur == regionFirst) continue;
            tmp.resize((size_t) (cur - regionFirst) * 3);
            int64_t w = 0;
            for (size_t j = runs.size(); j-- > 0;) {
                for (int64_t g0 = runs[j].first; g0 < runs[j].second;) {
                    const int64_t sum = (int64_t) triples[3 * g0 + 1] + triples[3 * g0 + 2];
                    int64_t g1 = g0 + 1;
                    while (g1 < runs[j].second && (int64_t) triples[3 * g1 + 1] + triples[3 * g1 + 2] == sum) g1++;
                    for (int64_t t = g1; t-- > g0;) {
                        memcpy(&tmp[3 * w], &triples[3 * t], 3 * sizeof(int32_t));
                        w++;
                    }
                    g0 = g1;
                }
            }
            memcpy(&triples[3 * regionFirst], tmp.data(), tmp.size() * sizeof(int32_t));
        }
    };
    const int64_t total = off[b->n];
    const int64_t nThreads = std::max<int64_t>(1, std::min<int64_t>({ (int64_t) std::thread::hardware_concurrency(), (int64_t) 16, total >> 20 }));
    if (nThreads <= 1) {
        reorder(0, nRegions);
        return CPB_OK;
    }
    /* cut the region list where a new pair starts, at about equal numbers of triples */
    std::vector<std::thread> pool;
    size_t r0 = 0;
    for (int64_t t = 0; t < nThreads && r0 < nRegions; t++) {
        size_t r1 = nRegions;
        if (t + 1 < nThreads) {
            const int64_t want = total * (t + 1) / nThreads;
            r1 = r0;
            while (r1 < nRegions && (off[b->hRegions[r1].pair] < want || (r1 > 0 && b->hRegions[r1].pair == b->hRegions[r1 - 1].pair))) r1++;
        }
        if (r1 > r0) pool.emplace_back(reorder, r0, r1);
        r0 = r1;
    }
    for (auto &t : pool) t.join();
    return CPB_OK;
}

/* device copies of the per-pair offsets the post-posterior kernels need: `off` (n+1 triple offsets of a list), xOff, yOff */
static int upload_pair_tables(cpb_batch *b, const std::vector<int64_t> &off, DevBuf &dOff, DevBuf &dX, DevBuf &dY) {
    int rc;
    const size_t bytes = (size_t) (b->n + 1) * sizeof(int64_t);
    if ((rc = dOff.reserve(bytes)) != CPB_OK || (rc = dX.reserve(bytes)) != CPB_OK || (rc = dY.reserve(bytes)) != CPB_OK) return rc;
    cudaStream_t st = b->ctx->stream;
    CUDA_TRY(cudaMemcpyAsync(dOff.p, off.data(), bytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dX.p, b->xOff.data(), bytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dY.p, b->yOff.data(), bytes, cudaMemcpyHostToDevice, st));
    return CPB_OK;
}

extern "C" int cpb_batch_reweight_pairs(cpb_batch *b, double gapGamma) {
    if (b == nullptr || (b->lastMode != CPB_MODE_ALIGNED_PAIRS && b->lastMode != CPB_MODE_ALIGNED_PAIRS_INDELS)) {
        cpb_set_error("cpb_batch_reweight_pairs: no aligned-pair results in this batch");
        return CPB_ERR_ARGUMENT;
    }
    if (!(gapGamma > 0.0) || b->outCount[0] == 0) return CPB_OK; /* reweightAlignedPairs2 returns its input for gapGamma <= 0 */
    if (b->reweighted) {
        cpb_set_error("cpb_batch_reweight_pairs: list 0 of this run has already been reweighted (the weights are rewritten in place; run the batch again first)");
        return CPB_ERR_ARGUMENT;
    }
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    DevBuf dOff, dX, dY, gX, gY;
    for (DevBuf *d : { &dOff, &dX, &dY, &gX, &gY }) d->pool = &b->ctx->pool;
    int rc = upload_pair_tables(b, b->pairOff[0], dOff, dX, dY);
    const int64_t lenX = b->xOff[b->n], lenY = b->yOff[b->n];
    if (rc == CPB_OK) rc = gX.reserve(std::max<int64_t>(lenX, 1) * sizeof(long long));
    if (rc == CPB_OK) rc = gY.reserve(std::max<int64_t>(lenY, 1) * sizeof(long long));
    if (rc == CPB_OK) {
        k_fill_i64<<<1184, 256, 0, st>>>(gX.as<long long>(), lenX, (long long) CPB_PAIR_ALIGNMENT_PROB_1);
        k_fill_i64<<<1184, 256, 0, st>>>(gY.as<long long>(), lenY, (long long) CPB_PAIR_ALIGNMENT_PROB_1);
        const int64_t nT = b->outCount[0];
        const unsigned grid = (unsigned) ((nT + 255) / 256);
        k_gap_weights<<<grid, 256, 0, st>>>(b->out[0].as<int32_t>(), nT, dOff.as<int64_t>(), (int) b->n, dX.as<int64_t>(), dY.as<int64_t>(),
                                            gX.as<long long>(), gY.as<long long>());
        k_reweight<<<grid, 256, 0, st>>>(b->out[0].as<int32_t>(), nT, dOff.as<int64_t>(), (int) b->n, dX.as<int64_t>(), dY.as<int64_t>(),
                                         gX.as<long long>(), gY.as<long long>(), gapGamma);
        b->stats.kernelLaunches += 4;
        cudaError_t e = cudaStreamSynchronize(st); /* the temporaries go back to the pool */
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) {
            cpb_set_error("cpb_batch_reweight_pairs: %s", cudaGetErrorString(e));
            rc = CPB_ERR_CUDA;
        } else {
            b->reweighted = true;
            b->stats.reweighted = 1;
            b->sunk[0] = false; /* a result sink holds the posteriors of the run, not these weights: the next fetch copies the list */
        }
    }
    for (DevBuf *d : { &dOff, &dX, &dY, &gX, &gY }) d->release();
    return rc;
}

extern "C" int cpb_batch_alignment_scores(cpb_batch *b, int64_t *scores) {
    if (b == nullptr || scores == nullptr || (b->lastMode != CPB_MODE_ALIGNED_PAIRS && b->lastMode != CPB_MODE_ALIGNED_PAIRS_INDELS)) {
        cpb_set_error("cpb_batch_alignment_scores: no aligned-pair results in this batch");
        return CPB_ERR_ARGUMENT;
    }
    if (b->n == 0) return CPB_OK;
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    DevBuf dOff, dX, dY, dS;
    for (DevBuf *d : { &dOff, &dX, &dY, &dS }) d->pool = &b->ctx->pool;
    int rc = upload_pair_tables(b, b->pairOff[0], dOff, dX, dY);
    if (rc == CPB_OK) rc = dS.reserve((size_t) b->n * sizeof(int64_t));
    if (rc == CPB_OK) {
        k_alignment_scores<<<(unsigned) ((b->n * 32 + 255) / 256), 256, 0, st>>>(b->out[0].as<int32_t>(), dOff.as<int64_t>(), (int) b->n, dX.as<int64_t>(),
                                                                              dY.as<int64_t>(), dS.as<int64_t>());
        b->stats.kernelLaunches++;
        cudaError_t e = cudaMemcpyAsync(scores, dS.p, (size_t) b->n * sizeof(int64_t), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) {
            cpb_set_error("cpb_batch_alignment_scores: %s", cudaGetErrorString(e));
            rc = CPB_ERR_CUDA;
        }
    }
    for (DevBuf *d : { &dOff, &dX, &dY, &dS }) d->release();
    return rc;
}

/* ------------------------------------------------------------------------------------------------
 * decoders on the device (decode_kernels.cuh): one alignment per pair from the lists of the last run, into the batch's alignment list.
 * The host functions of host/realign.c are the definition; libcpecan.so and cPecanRealign still decode on the host.
 * ---------------------------------------------------------------------------------------------- */
/* the pair descriptors of every pair (work offsets are filled in per chunk); false if a pair's list 0 is too long for the kernels' int32
 * indices */
static bool decode_pairs(const cpb_batch *b, bool withGaps, std::vector<DecodePair> &P) {
    P.assign((size_t) b->n, DecodePair());
    for (int64_t i = 0; i < b->n; i++) {
        DecodePair &D = P[(size_t) i];
        memset(&D, 0, sizeof(D));
        const int64_t n0 = b->pairOff[0][i + 1] - b->pairOff[0][i];
        if (n0 >= INT32_MAX) return false;
        D.list0 = b->pairOff[0][i];
        D.n0 = (int32_t) n0;
        if (withGaps) {
            D.gap1 = b->pairOff[1][i];
            D.n1 = (int32_t) (b->pairOff[1][i + 1] - b->pairOff[1][i]);
            D.gap2 = b->pairOff[2][i];
            D.n2 = (int32_t) (b->pairOff[2][i + 1] - b->pairOff[2][i]);
        }
        D.seqX = b->xOff[i];
        D.seqY = b->yOff[i];
        D.lX = (int32_t) (b->xOff[i + 1] - b->xOff[i]);
        D.lY = (int32_t) (b->yOff[i + 1] - b->yOff[i]);
    }
    return true;
}

/* Runs body(chunk) over chunks of pairs whose work arrays (workBytes(pair) each) and per-pair tables fit the scratch budget, and gathers
 * a per-pair list of triples: body launches the chunk's kernels and leaves every pair's length in chunk.lens; pair_chunks scans them into
 * chunk.off (the chunk's part of dOff, the n+1 device offsets of the list) and then calls emit(chunk), which writes the pairs' triples at
 * those offsets.  hostOff receives the offsets.  A single pair that does not fit returns CPB_ERR_MEMORY. */
struct DecodeChunk {
    int64_t p0, p1;
    int nC;
    DecodePair *desc;
    char *work;
    int32_t *lens, *aux;
    double *scores;
    int64_t *off;
};

template <class WorkBytes, class Body, class Emit>
static int pair_chunks(cpb_batch *b, const char *call, std::vector<DecodePair> &P, WorkBytes workBytes, Body body, Emit emit, double *scoresOut,
                       int64_t *dOff, std::vector<int64_t> &hostOff) {
    cpb_context *ctx = b->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = b->n;
    int rc;
    size_t budget = ctx->scratchBudget;
    if (budget == 0) {
        size_t freeB = 0, totalB = 0;
        CUDA_TRY(cudaMemGetInfo(&freeB, &totalB));
        budget = (size_t) ((double) (freeB + ctx->scratch.cap) * 0.70);
    }
    const size_t fixed = 16 * 256, perPair = sizeof(DecodePair) + 4 + 4 + 8 + 16;
    int64_t running = 0;
    if (n == 0) CUDA_TRY(cudaMemsetAsync(dOff, 0, sizeof(int64_t), st));
    for (int64_t p0 = 0; p0 < n;) {
        int64_t p1 = p0, W = 0;
        size_t bytes = fixed;
        while (p1 < n) {
            DecodePair &D = P[(size_t) p1];
            const size_t need = (size_t) workBytes(D) + perPair;
            if (fixed + need > budget) {
                cpb_set_error("%s: pair %lld (%d x %d, %d pairs in list 0) needs %zu bytes of scratch, more than the budget of %zu", call, (long long) p1, D.lX,
                              D.lY, D.n0, fixed + need, budget);
                return CPB_ERR_MEMORY;
            }
            if (bytes + need > budget || p1 - p0 >= (1 << 24)) break;
            bytes += need;
            D.work = W;
            W += (int64_t) workBytes(D);
            p1++;
        }
        DecodeChunk c;
        c.p0 = p0;
        c.p1 = p1;
        c.nC = (int) (p1 - p0);
        size_t at = 0;
        auto carve = [&](size_t nb) {
            const size_t here = at;
            at += (nb + 255) & ~(size_t) 255;
            return here;
        };
        const size_t oDesc = carve(c.nC * sizeof(DecodePair)), oLens = carve(c.nC * 4), oAux = carve(c.nC * 4), oScores = carve(c.nC * 8),
                     oTiles = carve(((c.nC + SCAN_TILE - 1) / SCAN_TILE + 1) * 8), oWork = carve((size_t) W);
        if ((rc = ctx->scratch.reserve(std::max<size_t>(at, 256))) != CPB_OK) return rc;
        char *s = ctx->scratch.as<char>();
        c.desc = reinterpret_cast<DecodePair *>(s + oDesc);
        c.lens = reinterpret_cast<int32_t *>(s + oLens);
        c.aux = reinterpret_cast<int32_t *>(s + oAux);
        c.scores = reinterpret_cast<double *>(s + oScores);
        c.work = s + oWork;
        c.off = dOff + p0;
        int64_t *dTiles = reinterpret_cast<int64_t *>(s + oTiles);
        CUDA_TRY(cudaMemcpyAsync(c.desc, P.data() + p0, c.nC * sizeof(DecodePair), cudaMemcpyHostToDevice, st));
        /* body and emit return the number of kernels they launched */
        b->stats.kernelLaunches += body(c);
        scan_counts(st, c.lens, c.nC, running, dTiles, c.off);
        b->stats.kernelLaunches += 3;
        b->stats.kernelLaunches += emit(c);
        CUDA_TRY(cudaGetLastError());
        if (scoresOut != nullptr) CUDA_TRY(cudaMemcpyAsync(scoresOut + p0, c.scores, c.nC * sizeof(double), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(&running, c.off + c.nC, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st)); /* the next chunk's scan starts from this total, and reuses the scratch */
        p0 = p1;
    }
    hostOff.assign((size_t) n + 1, 0);
    CUDA_TRY(cudaMemcpyAsync(hostOff.data(), dOff, (size_t) (n + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    return CPB_OK;
}

/* pair_chunks into the batch's alignment list */
template <class WorkBytes, class Body, class Emit>
static int decode_chunks(cpb_batch *b, const char *call, std::vector<DecodePair> &P, WorkBytes workBytes, Body body, Emit emit, double *scoresOut,
                         int64_t minCap = 0) {
    const int64_t n = b->n;
    int rc;
    int64_t cap = 0; /* every alignment is strictly increasing in x and y */
    for (int64_t i = 0; i < n; i++) cap += std::min(b->xOff[i + 1] - b->xOff[i], b->yOff[i + 1] - b->yOff[i]);
    cap = std::max(cap, minCap);
    DevBuf dOff;
    dOff.pool = &b->ctx->pool;
    if ((rc = b->aln.reserve((size_t) std::max<int64_t>(cap, 1) * 3 * sizeof(int32_t))) != CPB_OK || (rc = dOff.reserve((size_t) (n + 1) * sizeof(int64_t))) != CPB_OK)
        return rc;
    if ((rc = pair_chunks(b, call, P, workBytes, body, emit, scoresOut, dOff.as<int64_t>(), b->alnOff)) != CPB_OK) return rc;
    b->alnValid = true;
    return CPB_OK;
}

extern "C" int cpb_batch_ordered_chain(cpb_batch *b, float matchGamma) {
    if (b != nullptr) b->alnValid = false; /* a decode call replaces the list, also when it is refused */
    if (b == nullptr || (b->lastMode != CPB_MODE_ALIGNED_PAIRS && b->lastMode != CPB_MODE_ALIGNED_PAIRS_INDELS)) {
        cpb_set_error("cpb_batch_ordered_chain: no aligned-pair results in this batch");
        return CPB_ERR_ARGUMENT;
    }
    if (!(matchGamma >= 0.0f && matchGamma <= 1.0f)) {
        cpb_set_error("cpb_batch_ordered_chain: matchGamma must be in [0, 1] (a fraction of PAIR_ALIGNMENT_PROB_1), not %g", (double) matchGamma);
        return CPB_ERR_ARGUMENT;
    }
    std::vector<DecodePair> P;
    if (!decode_pairs(b, false, P)) {
        cpb_set_error("cpb_batch_ordered_chain: a pair has 2^31 or more aligned pairs");
        return CPB_ERR_ARGUMENT;
    }
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    const int32_t *list0 = b->out[0].as<int32_t>();
    return decode_chunks(
        b, "cpb_batch_ordered_chain", P, [](const DecodePair &D) { return chain_work_bytes(D.n0, D.lX, D.lY); },
        [&](DecodeChunk &c) {
            k_chain_sort<<<grid_of((int64_t) c.nC * 32, 256), 256, 0, st>>>(c.desc, c.nC, list0, c.work, (double) matchGamma);
            k_chain_sweep<<<grid_of((int64_t) c.nC * 32, 256), 256, 0, st>>>(c.desc, c.nC, c.work, c.lens, c.aux);
            return 2;
        },
        [&](DecodeChunk &c) {
            k_chain_write<<<grid_of(c.nC, 128), 128, 0, st>>>(c.desc, c.nC, c.work, c.lens, c.aux, c.off, b->aln.as<int32_t>());
            return 1;
        },
        nullptr);
}

/* The run's region and block tables, which put list 0 into the reference's order (what cpb_batch_fetch_pairs_reference_order does on the
 * host), on the device; every pair's range of regions into P. */
struct RefOrderTables {
    DevBuf tab;
    int64_t *shift = nullptr, *block0 = nullptr;
    int32_t *blocks = nullptr, *from = nullptr;
};

static int ref_order_tables(cpb_batch *b, std::vector<DecodePair> &P, RefOrderTables &T) {
    cudaStream_t st = b->ctx->stream;
    const int64_t nR = (int64_t) b->hRegions.size();
    std::vector<int64_t> regShift((size_t) std::max<int64_t>(nR, 1)), regBlock0((size_t) std::max<int64_t>(nR, 1));
    std::vector<int32_t> regBlocks((size_t) std::max<int64_t>(nR, 1)), blockFrom;
    int64_t nB = 0;
    for (int64_t r = 0; r < nR; r++) {
        const RegionDev &R = b->hRegions[(size_t) r];
        regShift[(size_t) r] = (int64_t) R.ox + R.oy - 2;
        regBlock0[(size_t) r] = nB;
        regBlocks[(size_t) r] = R.nBlocks;
        nB += R.nBlocks;
    }
    blockFrom.resize((size_t) std::max<int64_t>(nB, 1));
    for (int64_t k = 0; k < nB; k++) blockFrom[(size_t) k] = b->hBlocks[(size_t) k].from;
    for (int64_t r = nR; r-- > 0;) {
        DecodePair &D = P[(size_t) b->hRegions[(size_t) r].pair];
        if (D.region1 == 0) D.region1 = r + 1;
        D.region0 = r;
    }
    T.tab.pool = &b->ctx->pool;
    const size_t nRs = (size_t) std::max<int64_t>(nR, 1);
    const int rc = T.tab.reserve(nRs * 20 + blockFrom.size() * 4 + 64);
    if (rc != CPB_OK) return rc;
    T.shift = T.tab.as<int64_t>();
    T.block0 = T.shift + nRs;
    T.blocks = reinterpret_cast<int32_t *>(T.block0 + nRs);
    T.from = T.blocks + nRs;
    CUDA_TRY(cudaMemcpyAsync(T.shift, regShift.data(), nRs * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(T.block0, regBlock0.data(), nRs * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(T.blocks, regBlocks.data(), nRs * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(T.from, blockFrom.data(), blockFrom.size() * 4, cudaMemcpyHostToDevice, st));
    return CPB_OK;
}

extern "C" int cpb_batch_mea(cpb_batch *b, float gapGamma, int leftShift, double *scores) {
    if (b != nullptr) b->alnValid = false; /* a decode call replaces the list, also when it is refused */
    if (b == nullptr || b->lastMode != CPB_MODE_ALIGNED_PAIRS_INDELS) {
        cpb_set_error("cpb_batch_mea: needs the gap lists of an ALIGNED_PAIRS_INDELS run");
        return CPB_ERR_ARGUMENT;
    }
    if (!(gapGamma >= 0.0f && gapGamma <= FLT_MAX)) {
        cpb_set_error("cpb_batch_mea: gapGamma must be finite and >= 0, not %g", (double) gapGamma);
        return CPB_ERR_ARGUMENT;
    }
    std::vector<DecodePair> P;
    if (!decode_pairs(b, true, P)) {
        cpb_set_error("cpb_batch_mea: a pair has 2^31 or more aligned pairs");
        return CPB_ERR_ARGUMENT;
    }
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    RefOrderTables T;
    int rc = ref_order_tables(b, P, T);
    if (rc != CPB_OK) return rc;
    const int32_t *l0 = b->out[0].as<int32_t>(), *l1 = b->out[1].as<int32_t>(), *l2 = b->out[2].as<int32_t>();
    const uint8_t *kx = b->keptX.as<uint8_t>(), *ky = b->keptY.as<uint8_t>();
    return decode_chunks(
        b, "cpb_batch_mea", P, [](const DecodePair &D) { return mea_work_bytes(D.n0, D.lX, D.lY); },
        [&](DecodeChunk &c) {
            k_ref_order<<<grid_of(c.nC, 128), 128, 0, st>>>(c.desc, c.nC, l0, T.shift, T.block0, T.blocks, T.from, c.work);
            k_mea_gaps<<<grid_of((int64_t) c.nC * 32, 256), 256, 0, st>>>(c.desc, c.nC, l1, l2, c.work);
            k_mea<<<grid_of((int64_t) c.nC * 32, 256), 256, 0, st>>>(c.desc, c.nC, c.work, gapGamma, c.scores, c.lens);
            if (leftShift) k_decode_emit<true><<<grid_of(c.nC, 128), 128, 0, st>>>(c.desc, c.nC, c.work, kx, ky, c.lens, nullptr, nullptr);
            return leftShift ? 4 : 3;
        },
        [&](DecodeChunk &c) {
            if (leftShift) k_decode_emit<true><<<grid_of(c.nC, 128), 128, 0, st>>>(c.desc, c.nC, c.work, kx, ky, c.lens, c.off, b->aln.as<int32_t>());
            else k_decode_emit<false><<<grid_of(c.nC, 128), 128, 0, st>>>(c.desc, c.nC, c.work, kx, ky, c.lens, c.off, b->aln.as<int32_t>());
            return 1;
        },
        scores);
}

/* Test support, not part of the ABI header: the alignment list becomes list 0 of the last run in the reference's order as cpb_batch_mea
 * builds it on the device (k_ref_order), so that this permutation can be compared with cpb_batch_fetch_pairs_reference_order. */
extern "C" int cpb_debug_reference_order(cpb_batch *b) {
    if (b != nullptr) b->alnValid = false;
    if (b == nullptr || (b->lastMode != CPB_MODE_ALIGNED_PAIRS && b->lastMode != CPB_MODE_ALIGNED_PAIRS_INDELS)) {
        cpb_set_error("cpb_debug_reference_order: no aligned-pair results in this batch");
        return CPB_ERR_ARGUMENT;
    }
    std::vector<DecodePair> P;
    if (!decode_pairs(b, false, P)) {
        cpb_set_error("cpb_debug_reference_order: a pair has 2^31 or more aligned pairs");
        return CPB_ERR_ARGUMENT;
    }
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    RefOrderTables T;
    int rc = ref_order_tables(b, P, T);
    if (rc != CPB_OK) return rc;
    const int32_t *l0 = b->out[0].as<int32_t>();
    return decode_chunks(
        b, "cpb_debug_reference_order", P, [](const DecodePair &D) { return mea_work_bytes(D.n0, D.lX, D.lY); },
        [&](DecodeChunk &c) {
            k_ref_order<<<grid_of(c.nC, 128), 128, 0, st>>>(c.desc, c.nC, l0, T.shift, T.block0, T.blocks, T.from, c.work);
            k_ref_emit<<<grid_of(c.nC, 128), 128, 0, st>>>(c.desc, c.nC, c.work, c.lens, nullptr, nullptr);
            return 2;
        },
        [&](DecodeChunk &c) {
            k_ref_emit<<<grid_of(c.nC, 128), 128, 0, st>>>(c.desc, c.nC, c.work, c.lens, c.off, b->aln.as<int32_t>());
            return 1;
        },
        nullptr, b->outCount[0]);
}

extern "C" int64_t cpb_batch_alignments_count(const cpb_batch *b) { return b != nullptr && b->alnValid ? b->alnOff[(size_t) b->n] : 0; }

extern "C" int cpb_batch_fetch_alignments(const cpb_batch *b, int64_t *offsets, int32_t *triples) {
    if (b == nullptr || !b->alnValid || offsets == nullptr || (triples == nullptr && b->alnOff[(size_t) b->n] > 0)) {
        cpb_set_error("cpb_batch_fetch_alignments: %s", b != nullptr && !b->alnValid ? "no alignments: call cpb_batch_ordered_chain or cpb_batch_mea after the run"
                                                                                     : "bad argument");
        return CPB_ERR_ARGUMENT;
    }
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    memcpy(offsets, b->alnOff.data(), (size_t) (b->n + 1) * sizeof(int64_t));
    const int64_t count = b->alnOff[(size_t) b->n];
    if (count > 0) {
        CUDA_TRY(cudaMemcpyAsync(triples, b->aln.p, (size_t) count * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, b->ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(b->ctx->stream));
    }
    return CPB_OK;
}

extern "C" int cpb_batch_score_alignments(cpb_batch *b, int kind, double *scores) {
    if (b == nullptr || !b->alnValid || kind < CPB_SCORE_IDENTITY || kind > CPB_SCORE_POSTERIOR_IGNORING_GAPS || (scores == nullptr && b->n > 0)) {
        cpb_set_error("cpb_batch_score_alignments: %s", b != nullptr && !b->alnValid ? "no alignments: call cpb_batch_ordered_chain or cpb_batch_mea after the run"
                                                                                     : "bad argument (kind is one of CPB_SCORE_*)");
        return CPB_ERR_ARGUMENT;
    }
    if (b->n == 0) return CPB_OK;
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    DevBuf dOff, dX, dY, dS;
    for (DevBuf *d : { &dOff, &dX, &dY, &dS }) d->pool = &b->ctx->pool;
    int rc = upload_pair_tables(b, b->alnOff, dOff, dX, dY);
    if (rc != CPB_OK || (rc = dS.reserve((size_t) b->n * sizeof(double))) != CPB_OK) return rc;
    k_decode_scores<<<grid_of(b->n * 32, 256), 256, 0, st>>>(b->aln.as<int32_t>(), dOff.as<int64_t>(), (int) b->n, dX.as<int64_t>(), dY.as<int64_t>(),
                                                            b->keptX.as<uint8_t>(), b->keptY.as<uint8_t>(), kind, dS.as<double>());
    b->stats.kernelLaunches++;
    CUDA_TRY(cudaMemcpyAsync(scores, dS.p, (size_t) b->n * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    return CPB_OK;
}

/* The anchors job_prepare builds from the cigar of every pair's alignment (k_reanchor_count / k_reanchor_write), built into new buffers --
 * device triples, the device pair table, the page-locked host copy that build_regions reads -- which replace the batch's only once all of
 * them are there.  Only planning reads the anchors (k_split_flags, build_regions, k_band), so the lists, the alignment list and everything
 * else of the last run stay as they are; the kept plan goes. */
extern "C" int cpb_batch_anchors_from_alignments(cpb_batch *b, const CpbParams *p) {
    if (b == nullptr || p == nullptr || p->constraintDiagonalTrim < 0 || p->constraintDiagonalTrim > 0x7FFFFFFF || p->diagonalExpansion < 0 ||
        p->diagonalExpansion > 0x7FFFFFFF) {
        cpb_set_error("cpb_batch_anchors_from_alignments: %s", b == nullptr ? "bad argument"
                                                                            : (p == nullptr ? "no parameters" : "constraintDiagonalTrim and diagonalExpansion must be in [0, 2^31)"));
        return CPB_ERR_ARGUMENT;
    }
    if (!b->alnValid) {
        cpb_set_error("cpb_batch_anchors_from_alignments: no alignments: call cpb_batch_ordered_chain or cpb_batch_mea after the run");
        return CPB_ERR_ARGUMENT;
    }
    const int64_t n = b->n;
    std::vector<DecodePair> P((size_t) n);
    for (int64_t i = 0; i < n; i++) {
        DecodePair &D = P[(size_t) i];
        memset(&D, 0, sizeof(D));
        D.list0 = b->alnOff[(size_t) i];
        D.n0 = (int32_t) (b->alnOff[(size_t) i + 1] - b->alnOff[(size_t) i]); /* at most min(lX, lY) */
        D.seqX = b->xOff[(size_t) i];
        D.seqY = b->yOff[(size_t) i];
        D.lX = (int32_t) (b->xOff[(size_t) i + 1] - b->xOff[(size_t) i]);
        D.lY = (int32_t) (b->yOff[(size_t) i + 1] - b->yOff[(size_t) i]);
    }
    cpb_context *ctx = b->ctx;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    DevBuf tri, tab; /* the new device triples; the new pair table (aOff, xOff, yOff), whose first n + 1 entries the chunks fill */
    tri.pool = tab.pool = &ctx->pool;
    const size_t tabBytes = (size_t) (n + 1) * sizeof(int64_t);
    int rc;
    if ((rc = tri.reserve((size_t) std::max<int64_t>(b->alnOff[(size_t) n], 1) * 3 * sizeof(int32_t))) != CPB_OK || (rc = tab.reserve(3 * tabBytes)) != CPB_OK)
        return rc;
    const int32_t *aln = b->aln.as<int32_t>();
    const uint8_t *kx = b->keptX.as<uint8_t>(), *ky = b->keptY.as<uint8_t>();
    const int32_t trim = (int32_t) p->constraintDiagonalTrim, expansion = (int32_t) p->diagonalExpansion;
    std::vector<int64_t> aOff;
    rc = pair_chunks(
        b, "cpb_batch_anchors_from_alignments", P, [](const DecodePair &D) { return reanchor_work_bytes(D.n0); },
        [&](DecodeChunk &c) {
            k_reanchor_count<<<grid_of((int64_t) c.nC * 32, 256), 256, 0, st>>>(c.desc, c.nC, aln, kx, ky, c.work, trim, c.lens);
            return 1;
        },
        [&](DecodeChunk &c) {
            k_reanchor_write<<<grid_of((int64_t) c.nC * 32, 256), 256, 0, st>>>(c.desc, c.nC, aln, c.work, expansion, c.off, tri.as<int32_t>());
            return 1;
        },
        nullptr, tab.as<int64_t>(), aOff);
    if (rc != CPB_OK) return rc;
    if (n > 0) CUDA_TRY(cudaMemcpyAsync(tab.as<char>() + tabBytes, b->dPairTab.as<char>() + tabBytes, 2 * tabBytes, cudaMemcpyDeviceToDevice, st));
    const int64_t nA = aOff[(size_t) n];
    const size_t bytes = (size_t) (3 * nA) * sizeof(int32_t);
    int32_t *host = nA > 0 ? static_cast<int32_t *>(ctx->pinned.take(bytes)) : nullptr;
    std::vector<int32_t> own;
    if (nA > 0 && host == nullptr) {
        own.resize((size_t) (3 * nA));
        host = own.data();
    }
    cudaError_t e = nA > 0 ? cudaMemcpyAsync(host, tri.p, bytes, cudaMemcpyDeviceToHost, st) : cudaSuccess;
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        if (host != nullptr && own.empty()) ctx->pinned.give(host);
        cpb_set_error("cpb_batch_anchors_from_alignments: %s", cudaGetErrorString(e));
        return CPB_ERR_CUDA;
    }
    /* everything is built: swap */
    if (b->anchors != nullptr && b->anchorsOwn.empty()) ctx->pinned.give(b->anchors);
    b->anchors = host;
    b->anchorsOwn.swap(own);
    b->aOff.swap(aOff);
    b->dAnchors.release();
    b->dAnchors.adopt(tri);
    if (n > 0) {
        b->dPairTab.release();
        b->dPairTab.adopt(tab);
    }
    b->oddExpansionPair = -1;
    if (expansion & 1) {
        for (int64_t i = 0; i < n && b->oddExpansionPair < 0; i++)
            if (b->aOff[(size_t) i + 1] > b->aOff[(size_t) i]) b->oddExpansionPair = i;
    }
    b->planValid = false;
    return CPB_OK;
}

extern "C" int cpb_batch_fetch_expectations(cpb_batch *b, double *perPair, double *total) {
    if (b == nullptr || b->lastMode != CPB_MODE_EXPECTATIONS) {
        cpb_set_error("cpb_batch_fetch_expectations: last run was not in expectation mode");
        return CPB_ERR_ARGUMENT;
    }
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    const int len = CPB_HMM_LEN(b->lastS);
    if (perPair && b->n > 0) CUDA_TRY(cudaMemcpyAsync(perPair, b->perPair.p, (size_t) b->n * len * sizeof(double), cudaMemcpyDeviceToHost, b->ctx->stream));
    if (total) CUDA_TRY(cudaMemcpyAsync(total, b->hmmTotal.p, len * sizeof(double), cudaMemcpyDeviceToHost, b->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(b->ctx->stream));
    return CPB_OK;
}

/* ------------------------------------------------------------------------------------------------
 * EM reduction across the GPUs of one process: every batch's expectation total (CPB_HMM_LEN(S) doubles in its device's HBM) becomes
 * the sum over all batches, by ONE ncclAllReduce(ncclDouble, ncclSum) per device inside a group call -- the replacement of
 * cPecanEm.py:182-188, which sums per-job expectation files.  NCCL is bound at run time (dlopen of libnccl.so.2: the library has no
 * link-time dependency on it); without it the caller adds the 58 / 106 doubles up on the host.
 * ---------------------------------------------------------------------------------------------- */
#include <dlfcn.h>
namespace {
struct Nccl {
    typedef void *Comm;
    int (*commInitAll)(Comm *, int, const int *) = nullptr;
    int (*commDestroy)(Comm) = nullptr;
    int (*allReduce)(const void *, void *, size_t, int, int, Comm, cudaStream_t) = nullptr;
    int (*groupStart)() = nullptr;
    int (*groupEnd)() = nullptr;
    const char *(*errorString)(int) = nullptr;
    bool tried = false, ok = false;
    std::vector<int> devices; /* the communicators below were made for exactly these devices, in this order */
    std::vector<Comm> comms;
    bool load() {
        if (tried) return ok;
        tried = true;
        void *h = nullptr;
        for (const char *name : { "libnccl.so.2", "libnccl.so" }) {
            if ((h = dlopen(name, RTLD_NOW | RTLD_LOCAL)) != nullptr) break;
        }
        if (h == nullptr) return false;
        commInitAll = (int (*)(Comm *, int, const int *)) dlsym(h, "ncclCommInitAll");
        commDestroy = (int (*)(Comm)) dlsym(h, "ncclCommDestroy");
        allReduce = (int (*)(const void *, void *, size_t, int, int, Comm, cudaStream_t)) dlsym(h, "ncclAllReduce");
        groupStart = (int (*)()) dlsym(h, "ncclGroupStart");
        groupEnd = (int (*)()) dlsym(h, "ncclGroupEnd");
        errorString = (const char *(*) (int) ) dlsym(h, "ncclGetErrorString");
        ok = commInitAll && commDestroy && allReduce && groupStart && groupEnd && errorString;
        return ok;
    }
} g_nccl;
} // namespace

extern "C" int cpb_expectations_allreduce(cpb_batch *const *batches, int n) {
    if (batches == nullptr || n < 1) {
        cpb_set_error("cpb_expectations_allreduce: bad argument");
        return CPB_ERR_ARGUMENT;
    }
    std::vector<int> devices;
    for (int i = 0; i < n; i++) {
        if (batches[i] == nullptr || batches[i]->lastMode != CPB_MODE_EXPECTATIONS || batches[i]->lastS != batches[0]->lastS) {
            cpb_set_error("cpb_expectations_allreduce: batch %d has no expectations of the same model", i);
            return CPB_ERR_ARGUMENT;
        }
        devices.push_back(batches[i]->ctx->device);
    }
    if (n == 1) return CPB_OK;
    for (int i = 0; i < n; i++) {
        for (int j = 0; j < i; j++) {
            if (devices[i] == devices[j]) {
                cpb_set_error("cpb_expectations_allreduce: batches %d and %d are on the same device", j, i);
                return CPB_ERR_ARGUMENT;
            }
        }
    }
    if (!g_nccl.load()) {
        cpb_set_error("cpb_expectations_allreduce: NCCL (libnccl.so.2) is not available");
        return CPB_ERR_CUDA;
    }
    if (g_nccl.devices != devices) {
        for (auto c : g_nccl.comms) g_nccl.commDestroy(c);
        g_nccl.comms.assign(n, nullptr);
        g_nccl.devices.clear();
        const int rc = g_nccl.commInitAll(g_nccl.comms.data(), n, devices.data());
        if (rc != 0) {
            cpb_set_error("ncclCommInitAll: %s", g_nccl.errorString(rc));
            g_nccl.comms.clear();
            return CPB_ERR_CUDA;
        }
        g_nccl.devices = devices;
    }
    const size_t len = CPB_HMM_LEN(batches[0]->lastS);
    int rc = g_nccl.groupStart();
    for (int i = 0; i < n && rc == 0; i++) {
        cudaSetDevice(devices[i]);
        rc = g_nccl.allReduce(batches[i]->hmmTotal.p, batches[i]->hmmTotal.p, len, /* ncclDouble */ 8, /* ncclSum */ 0, g_nccl.comms[i], batches[i]->ctx->stream);
    }
    const int rcEnd = g_nccl.groupEnd();
    if (rc == 0) rc = rcEnd;
    if (rc != 0) {
        cpb_set_error("ncclAllReduce: %s", g_nccl.errorString(rc));
        return CPB_ERR_CUDA;
    }
    for (int i = 0; i < n; i++) {
        CUDA_TRY(cudaSetDevice(devices[i]));
        CUDA_TRY(cudaStreamSynchronize(batches[i]->ctx->stream));
    }
    return CPB_OK;
}

extern "C" const double *cpb_batch_device_expectation_total(const cpb_batch *b) {
    return (b && b->lastMode == CPB_MODE_EXPECTATIONS) ? b->hmmTotal.as<double>() : nullptr;
}

extern "C" int cpb_batch_fetch_forward(cpb_batch *b, double *logProb) {
    if (b == nullptr || b->lastMode != CPB_MODE_FORWARD || logProb == nullptr) {
        cpb_set_error("cpb_batch_fetch_forward: last run was not in forward mode");
        return CPB_ERR_ARGUMENT;
    }
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    if (b->n > 0) {
        CUDA_TRY(cudaMemcpyAsync(logProb, b->forwardOut.p, (size_t) b->n * sizeof(double), cudaMemcpyDeviceToHost, b->ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(b->ctx->stream));
    }
    return CPB_OK;
}

/* ------------------------------------------------------------------------------------------------
 * cpb_band: run the device band builder on one problem and copy the band back (unit-test / inspection entry)
 * ---------------------------------------------------------------------------------------------- */
extern "C" int cpb_band(cpb_context *ctx, const int64_t *anchors, int64_t nAnchors, int64_t lX, int64_t lY, int64_t expansion, int dynamic,
                        int64_t *out3) {
    if (ctx == nullptr || lX < 0 || lY < 0 || out3 == nullptr) return CPB_ERR_ARGUMENT;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int64_t N = lX + lY;
    DevBuf dRegion, dDiags, dBlocks, dAnch, dStrips;
    int rc;
    if ((rc = dRegion.reserve(sizeof(RegionDev))) != CPB_OK || (rc = dDiags.reserve((N + 3) * sizeof(DiagRec))) != CPB_OK ||
        (rc = dBlocks.reserve(sizeof(BlockRec))) != CPB_OK || (rc = dAnch.reserve(std::max<int64_t>(nAnchors, 1) * 3 * sizeof(int32_t))) != CPB_OK)
        return rc;
    std::vector<int32_t> a32(3 * std::max<int64_t>(nAnchors, 1), 0);
    for (int64_t i = 0; i < 3 * nAnchors; i++) a32[i] = (int32_t) anchors[i];
    RegionDev R;
    memset(&R, 0, sizeof(R));
    R.lX = (int32_t) lX;
    R.lY = (int32_t) lY;
    R.nAnchors = (int32_t) nAnchors;
    R.blockCap = 0;
    cudaStream_t st = ctx->stream;
    CUDA_TRY(cudaMemcpyAsync(dAnch.p, a32.data(), a32.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dRegion.p, &R, sizeof(R), cudaMemcpyHostToDevice, st));
    BandArgs ba;
    memset(&ba, 0, sizeof(ba));
    ba.regions = dRegion.as<RegionDev>();
    ba.anchors = dAnch.as<int32_t>();
    ba.diags = dDiags.as<DiagRec>();
    if ((rc = dStrips.reserve(((lX >> 5) + 1) * sizeof(StripRec))) != CPB_OK) return rc;
    ba.blocks = dBlocks.as<BlockRec>();
    ba.strips = dStrips.as<StripRec>();
    ba.nRegions = 1;
    ba.expansion = (int32_t) expansion;
    ba.dynamic = dynamic;
    ba.minDiags = 2;
    ba.traceBack = 1;
    ba.scheduleOn = 0;
    k_band<<<1, 32 * BAND_WARPS, 0, st>>>(ba);
    std::vector<DiagRec> recs(N + 2);
    CUDA_TRY(cudaMemcpyAsync(recs.data(), dDiags.p, (N + 2) * sizeof(DiagRec), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&R, dRegion.p, sizeof(R), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    dRegion.release();
    dDiags.release();
    dBlocks.release();
    dAnch.release();
    dStrips.release();
    for (int64_t d = 0; d <= N; d++) {
        out3[3 * d] = d;
        out3[3 * d + 1] = recs[d].xmyL;
        out3[3 * d + 2] = recs[d].xmyL + 2 * ((int64_t) recs[d].width - 1);
    }
    if (R.err != 0) {
        cpb_set_error("cpb_band: anchors produce an invalid band diagonal");
        return CPB_ERR_BAND;
    }
    return CPB_OK;
}
