"""ctypes binding of include/cpecan_b200.h.

Names follow the reference's C API so tests read like cPecan's own
(tests/pairwiseAlignerTest.c): ``getAlignedPairsUsingAnchors(sM, sX, sY, anchorPairs, p, l, r)``
(inc/pairwiseAligner.h:75), ``getExpectationsUsingAnchors`` (:105), ``computeForwardProbability`` (:56),
``stateMachine5_construct`` / ``hmm_getStateMachine`` (inc/stateMachine.h:95-99).
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CPB_LIB") or os.path.join(_HERE, "lib", "libcpecan_b200.so")  # CPB_LIB: kernel-variant experiments only

PAIR_ALIGNMENT_PROB_1 = 10000000
fiveState, fiveStateAsymmetric, threeState, threeStateAsymmetric = 0, 1, 2, 3
MODE_ALIGNED_PAIRS, MODE_ALIGNED_PAIRS_INDELS, MODE_EXPECTATIONS, MODE_FORWARD = 0, 1, 2, 3
SCORE_IDENTITY, SCORE_IDENTITY_IGNORING_GAPS, SCORE_POSTERIOR, SCORE_POSTERIOR_IGNORING_GAPS = 0, 1, 2, 3
OP_MATCH, OP_INDEL_X, OP_INDEL_Y = 0, 1, 2  # cigar operation types (CPB_OP_*)


class CpbError(RuntimeError):
    pass


class CpbParams(C.Structure):
    """PairwiseAlignmentParameters (inc/pairwiseAligner.h:28-41)."""

    _fields_ = [
        ("threshold", C.c_double),
        ("minDiagsBetweenTraceBack", C.c_int64),
        ("traceBackDiagonals", C.c_int64),
        ("diagonalExpansion", C.c_int64),
        ("constraintDiagonalTrim", C.c_int64),
        ("anchorMatrixBiggerThanThis", C.c_int64),
        ("repeatMaskMatrixBiggerThanThis", C.c_int64),
        ("splitMatrixBiggerThanThis", C.c_int64),
        ("alignAmbiguityCharacters", C.c_int32),
        ("gapGamma", C.c_float),
        ("dynamicAnchorExpansion", C.c_int32),
        ("pad_", C.c_int32),
    ]


class CpbModel(C.Structure):
    _fields_ = [
        ("type", C.c_int32),
        ("stateNumber", C.c_int32),
        ("start", C.c_double * 5),
        ("raggedStart", C.c_double * 5),
        ("end", C.c_double * 5),
        ("raggedEnd", C.c_double * 5),
        ("tLower", C.c_double * 4),
        ("tMiddle", C.c_double * 5),
        ("tUpper", C.c_double * 4),
        ("eMatch", C.c_double * 25),
        ("eGapX", C.c_double * 5),
        ("eGapY", C.c_double * 5),
    ]


class CpbRunStats(C.Structure):
    _fields_ = [
        ("nPairs", C.c_int64),
        ("nRegions", C.c_int64),
        ("nBlocks", C.c_int64),
        ("nChunks", C.c_int64),
        ("cells", C.c_int64),
        ("diagonals", C.c_int64),
        ("outputTriples", C.c_int64),
        ("kernelLaunches", C.c_int64),
        ("msBand", C.c_double),
        ("msForward", C.c_double),
        ("msBackward", C.c_double),
        ("msTotals", C.c_double),
        ("msPosterior", C.c_double),
        ("maxWidth", C.c_int32),
        ("twoPass", C.c_int32),
        ("msCheckpoint", C.c_double),
        ("pintFixups", C.c_int64),
        ("planReused", C.c_int64),
        ("reweighted", C.c_int64),
    ]


def hmm_len(S):
    return S * S + S * 16 + 1


def _require_built():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libcpecan_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -f cpecan_b200/csrc/Makefile`. There is no CPU fallback." % LIB_PATH
        )


_require_built()  # importing the package without the built library fails here, loudly


def _load():
    _require_built()
    L = C.CDLL(LIB_PATH)
    P = C.POINTER
    L.cpb_version.restype = C.c_char_p
    L.cpb_last_error.restype = C.c_char_p
    L.cpb_params_default.argtypes = [P(CpbParams)]
    L.cpb_model_default.argtypes = [C.c_int, P(CpbModel)]
    L.cpb_model_from_hmm.argtypes = [C.c_int, P(C.c_double), P(C.c_double), P(CpbModel)]
    L.cpb_split_points.restype = C.c_int64
    L.cpb_split_points.argtypes = [P(C.c_int64), C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, P(C.c_int64), C.c_int64]
    L.cpb_context_create.argtypes = [C.c_int, C.c_void_p, P(C.c_void_p)]
    L.cpb_context_destroy.argtypes = [C.c_void_p]
    L.cpb_context_set_scratch_budget.argtypes = [C.c_void_p, C.c_size_t]
    L.cpb_band.argtypes = [C.c_void_p, P(C.c_int64), C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, P(C.c_int64)]
    L.cpb_batch_create.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, P(C.c_void_p)]
    L.cpb_batch_create_anchored.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            P(CpbParams), P(C.c_void_p)]
    L.cpb_batch_create_from_cigars.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p, P(CpbParams), P(C.c_void_p)]
    L.cpb_batch_anchor_count.restype = C.c_int64
    L.cpb_batch_anchor_count.argtypes = [C.c_void_p]
    L.cpb_batch_fetch_anchors.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.cpb_batch_destroy.argtypes = [C.c_void_p]
    L.cpb_batch_run.argtypes = [C.c_void_p, P(CpbModel), P(CpbParams), C.c_int]
    L.cpb_batch_stats.argtypes = [C.c_void_p, P(CpbRunStats)]
    L.cpb_batch_result_count.restype = C.c_int64
    L.cpb_batch_result_count.argtypes = [C.c_void_p, C.c_int]
    L.cpb_batch_fetch_pairs.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.cpb_batch_set_result_sink.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]
    L.cpb_batch_fetch_pairs_reference_order.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.cpb_batch_reweight_pairs.argtypes = [C.c_void_p, C.c_double]
    L.cpb_batch_alignment_scores.argtypes = [C.c_void_p, C.c_void_p]
    L.cpb_batch_ordered_chain.argtypes = [C.c_void_p, C.c_float]
    L.cpb_batch_mea.argtypes = [C.c_void_p, C.c_float, C.c_int, C.c_void_p]
    L.cpb_batch_alignments_count.restype = C.c_int64
    L.cpb_batch_alignments_count.argtypes = [C.c_void_p]
    L.cpb_batch_fetch_alignments.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.cpb_batch_score_alignments.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.cpb_batch_anchors_from_alignments.argtypes = [C.c_void_p, P(CpbParams)]
    L.cpb_batch_alignment_cigars.argtypes = [C.c_void_p, C.c_void_p]
    L.cpb_batch_fetch_cigars.argtypes = [C.c_void_p, C.c_void_p]
    L.cpb_batch_alignments_from_cigars.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
    L.cpb_batch_device_triples.restype = C.c_void_p
    L.cpb_batch_device_triples.argtypes = [C.c_void_p, C.c_int]
    L.cpb_batch_fetch_expectations.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.cpb_batch_device_expectation_total.restype = C.c_void_p
    L.cpb_batch_device_expectation_total.argtypes = [C.c_void_p]
    L.cpb_batch_fetch_forward.argtypes = [C.c_void_p, C.c_void_p]
    return L


class _LazyLib:
    """The shared library is mapped on first use, not on import: `import cpecan_b200` (for the synthetic-data generator, say) must not
    put libcpecan_b200.so into a process that then only runs the CPU reference (bench.py --impl reference)."""

    _lib = None

    def __getattr__(self, name):
        if _LazyLib._lib is None:
            _LazyLib._lib = _load()
        return getattr(_LazyLib._lib, name)


lib = _LazyLib()


def _check(rc):
    if rc != 0:
        raise CpbError("cpecan_b200 error %d: %s" % (rc, lib.cpb_last_error().decode()))


# ---- parameters and models (host side, no GPU needed) ----
def pairwiseAlignmentBandingParameters_construct():
    p = CpbParams()
    lib.cpb_params_default(C.byref(p))
    return p


def stateMachine5_construct(type_=fiveState):
    if type_ not in (fiveState, fiveStateAsymmetric):
        raise CpbError("Wrong type for five state %d" % type_)
    m = CpbModel()
    _check(lib.cpb_model_default(type_, C.byref(m)))
    return m


def stateMachine3_construct(type_=threeState):
    if type_ not in (threeState, threeStateAsymmetric):
        raise CpbError("Tried to create a three state state-machine with the wrong type")
    m = CpbModel()
    _check(lib.cpb_model_default(type_, C.byref(m)))
    return m


def hmm_getStateMachine(type_, transitions, emissions):
    """hmm_getStateMachine (impl/stateMachine.c:797): transitions S*S, emissions S*16 probabilities."""
    t = np.ascontiguousarray(transitions, dtype=np.float64).ravel()
    e = np.ascontiguousarray(emissions, dtype=np.float64).ravel()
    m = CpbModel()
    _check(lib.cpb_model_from_hmm(type_, t.ctypes.data_as(C.POINTER(C.c_double)), e.ctypes.data_as(C.POINTER(C.c_double)), C.byref(m)))
    return m


def _anchor_array(anchorPairs):
    a = np.ascontiguousarray(anchorPairs, dtype=np.int64).reshape(-1)
    if a.size % 3 != 0:
        # allow (x, y) pairs: expansion 0
        a2 = a.reshape(-1, 2)
        a = np.concatenate([a2, np.zeros((a2.shape[0], 1), dtype=np.int64)], axis=1).reshape(-1)
    return a


def getSplitPoints(anchorPairs, lX, lY, splitMatrixBiggerThanThis, raggedLeft, raggedRight):
    a = _anchor_array(anchorPairs)
    n = a.size // 3
    cap = n + 2
    out = np.zeros(4 * cap, dtype=np.int64)
    k = lib.cpb_split_points(a.ctypes.data_as(C.POINTER(C.c_int64)) if n else None, n, lX, lY, splitMatrixBiggerThanThis,
                             int(raggedLeft), int(raggedRight), out.ctypes.data_as(C.POINTER(C.c_int64)), cap)
    return [tuple(int(v) for v in out[4 * i:4 * i + 4]) for i in range(k)]


# ---- device objects ----
class Context:
    def __init__(self, device=0, stream=None):
        h = C.c_void_p()
        _check(lib.cpb_context_create(device, C.c_void_p(stream) if stream else None, C.byref(h)))
        self.h = h
        self.device = device

    def set_scratch_budget(self, nbytes):
        lib.cpb_context_set_scratch_budget(self.h, int(nbytes))

    def band(self, anchorPairs, lX, lY, expansion, dynamic=False):
        a = _anchor_array(anchorPairs)
        n = a.size // 3
        out = np.zeros(3 * (lX + lY + 1), dtype=np.int64)
        _check(lib.cpb_band(self.h, a.ctypes.data_as(C.POINTER(C.c_int64)) if n else None, n, lX, lY, expansion, int(dynamic),
                            out.ctypes.data_as(C.POINTER(C.c_int64))))
        return out.reshape(-1, 3)

    def close(self):
        if self.h:
            lib.cpb_context_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = None


def default_context():
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(int(os.environ.get("LOCAL_RANK", "0")) if os.environ.get("CPB_USE_LOCAL_RANK") else 0)
    return _default_ctx


def _as_bytes(s):
    return s.encode() if isinstance(s, str) else bytes(s)


def _pack_sequences(seqs):
    """-> (concatenated uint8 bytes, int64 offsets[n+1])"""
    s = [_as_bytes(q) for q in seqs]
    off = np.zeros(len(s) + 1, dtype=np.int64)
    np.cumsum([len(q) for q in s], out=off[1:])
    return np.frombuffer(b"".join(s) + b"\0", dtype=np.uint8), off


def _ragged(flags):
    return np.ascontiguousarray(flags, dtype=np.uint8) if flags is not None else None


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else None


def _cigar_arrays(cigars):
    """(offsets[n+1], ops[m, 2]) as Batch.alignment_cigars returns them -> contiguous int64 offsets and int32 operations"""
    off, ops = cigars
    return np.ascontiguousarray(off, dtype=np.int64), np.ascontiguousarray(np.asarray(ops).reshape(-1, 2), dtype=np.int32)


class Batch:
    """n independent (seqX, seqY, anchors, ragged flags) problems resident on the device."""

    def __init__(self, ctx, seqsX, seqsY, anchors=None, raggedLeft=None, raggedRight=None, packed=None):
        self.ctx = ctx
        if packed is not None:
            # packed = dict(seqX=uint8 array, xOff=int64, seqY=..., yOff=..., anchors=int64 triples (flat), aOff=int64, rl, rr)
            self.n = len(packed["xOff"]) - 1
            bx, xo, by, yo = packed["seqX"], packed["xOff"], packed["seqY"], packed["yOff"]
            an, ao = packed["anchors"], packed["aOff"]
            rl, rr = packed.get("rl"), packed.get("rr")
        else:
            self.n = len(seqsX)
            bx, xo = _pack_sequences(seqsX)
            by, yo = _pack_sequences(seqsY)
            alist = [_anchor_array(a) for a in (anchors if anchors is not None else [[]] * self.n)]
            ao = np.zeros(self.n + 1, dtype=np.int64)
            np.cumsum([a.size // 3 for a in alist], out=ao[1:])
            an = np.concatenate(alist) if alist and ao[-1] > 0 else np.zeros(3, dtype=np.int64)
            rl, rr = _ragged(raggedLeft), _ragged(raggedRight)
        self._keep = (bx, xo, by, yo, an, ao, rl, rr)
        h = C.c_void_p()
        _check(lib.cpb_batch_create(ctx.h, self.n, _ptr(bx), _ptr(xo), _ptr(by), _ptr(yo), _ptr(an), _ptr(ao), _ptr(rl), _ptr(rr), C.byref(h)))
        self.h = h
        self.S = None

    @classmethod
    def anchored(cls, ctx, seqsX, seqsY, params, raggedLeft=None, raggedRight=None):
        """A batch whose anchors the device finds from the raw sequences: per pair the triples libcpecan.so's
        getBlastPairsForPairwiseAlignmentParameters returns for `params` (lower case is the soft mask)."""
        self = cls.__new__(cls)
        self.ctx, self.n, self.S, self.h = ctx, len(seqsX), None, None
        bx, xo = _pack_sequences(seqsX)
        by, yo = _pack_sequences(seqsY)
        rl, rr = _ragged(raggedLeft), _ragged(raggedRight)
        h = C.c_void_p()
        _check(lib.cpb_batch_create_anchored(ctx.h, self.n, _ptr(bx), _ptr(xo), _ptr(by), _ptr(yo), _ptr(rl), _ptr(rr), C.byref(params), C.byref(h)))
        self.h = h
        return self

    @classmethod
    def from_cigars(cls, ctx, seqsX, seqsY, cigars, params, raggedLeft=None, raggedRight=None):
        """A batch whose anchors the device builds from one forward-strand cigar per pair, cigars = (offsets[n+1] int64, ops[m, 2] int32
        (type OP_*, length)) as alignment_cigars returns them: the anchors cPecanRealign's job_prepare keeps for that alignment under
        params.constraintDiagonalTrim and params.diagonalExpansion"""
        self = cls.__new__(cls)
        self.ctx, self.n, self.S, self.h = ctx, len(seqsX), None, None
        bx, xo = _pack_sequences(seqsX)
        by, yo = _pack_sequences(seqsY)
        oo, ops = _cigar_arrays(cigars)
        rl, rr = _ragged(raggedLeft), _ragged(raggedRight)
        h = C.c_void_p()
        _check(lib.cpb_batch_create_from_cigars(ctx.h, self.n, _ptr(bx), _ptr(xo), _ptr(by), _ptr(yo), _ptr(oo), _ptr(ops) if len(ops) else None,
                                                _ptr(rl), _ptr(rr), C.byref(params) if params is not None else None, C.byref(h)))
        self.h = h
        return self

    def fetch_anchors(self):
        """-> (offsets[n+1] int64, triples[m, 3] int64 (x, y, expansion)): the anchors the batch holds, the caller's or the device's"""
        m = int(lib.cpb_batch_anchor_count(self.h))
        off = np.zeros(self.n + 1, dtype=np.int64)
        tri = np.zeros((max(m, 1), 3), dtype=np.int64)
        _check(lib.cpb_batch_fetch_anchors(self.h, C.c_void_p(off.ctypes.data), C.c_void_p(tri.ctypes.data)))
        return off, tri[:m]

    def run(self, model, params, mode):
        self.S = model.stateNumber
        _check(lib.cpb_batch_run(self.h, C.byref(model), C.byref(params), mode))

    def stats(self):
        s = CpbRunStats()
        lib.cpb_batch_stats(self.h, C.byref(s))
        return s

    def result_count(self, which=0):
        return int(lib.cpb_batch_result_count(self.h, which))

    def fetch_pairs(self, which=0, out=None, reference_order=False):
        """-> (offsets[n+1], triples[count,3] int32 (pInt, x, y)); per pair sorted by (x+y, x), or with reference_order in the
        order the reference's own lists have (what libcpecan.so returns)"""
        cnt = self.result_count(which)
        off = np.zeros(self.n + 1, dtype=np.int64)
        tri = out if out is not None else np.zeros((max(cnt, 1), 3), dtype=np.int32)
        fetch = lib.cpb_batch_fetch_pairs_reference_order if reference_order else lib.cpb_batch_fetch_pairs
        _check(fetch(self.h, which, C.c_void_p(off.ctypes.data), C.c_void_p(tri.ctypes.data)))
        return off, tri[:cnt]

    def set_result_sink(self, which, out):
        """out: int32 array [capacity, 3] in page-locked host memory that the next runs fill with list `which` while they compute;
        fetch_pairs(which, out=out) then only returns the offsets (None removes the sink)"""
        if out is None:
            _check(lib.cpb_batch_set_result_sink(self.h, which, None, 0))
        else:
            assert out.dtype == np.int32 and out.flags["C_CONTIGUOUS"]
            _check(lib.cpb_batch_set_result_sink(self.h, which, C.c_void_p(out.ctypes.data), out.shape[0]))
        self._sink = out

    def reweight_pairs(self, gap_gamma):
        """reweightAlignedPairs2 (impl/pairwiseAligner.c:1519-1560) on the device, in place on list 0"""
        _check(lib.cpb_batch_reweight_pairs(self.h, float(gap_gamma)))

    def alignment_scores(self):
        """getAlignmentScore (impl/multipleAligner.c:604-619) per pair -> int64[n]"""
        out = np.zeros(self.n, dtype=np.int64)
        _check(lib.cpb_batch_alignment_scores(self.h, C.c_void_p(out.ctypes.data)))
        return out

    def ordered_chain(self, match_gamma):
        """filterPairwiseAlignmentToMakePairsOrdered (impl/multipleAligner.c:945-972) of every pair's list 0, on the device, into the
        batch's alignment list (fetch_alignments)"""
        _check(lib.cpb_batch_ordered_chain(self.h, float(match_gamma)))

    def mea(self, gap_gamma, left_shift=True):
        """getMaximalExpectedAccuracyPairwiseAlignment (impl/pairwiseAligner.c:1603-1724), and with left_shift leftShiftAlignment
        (:1726-1767), of every pair of an ALIGNED_PAIRS_INDELS run, on the device, into the alignment list -> alignmentScore float64[n]"""
        out = np.zeros(max(self.n, 1), dtype=np.float64)
        _check(lib.cpb_batch_mea(self.h, float(gap_gamma), int(bool(left_shift)), C.c_void_p(out.ctypes.data)))
        return out[: self.n]

    def fetch_alignments(self):
        """-> (offsets[n+1] int64, triples[count, 3] int32 (pInt, x, y)): the alignment list of the last decode call"""
        m = int(lib.cpb_batch_alignments_count(self.h))
        off = np.zeros(self.n + 1, dtype=np.int64)
        tri = np.zeros((max(m, 1), 3), dtype=np.int32)
        _check(lib.cpb_batch_fetch_alignments(self.h, C.c_void_p(off.ctypes.data), C.c_void_p(tri.ctypes.data)))
        return off, tri[:m]

    def score_alignments(self, kind):
        """scoreByIdentity / ...IgnoringGaps / scoreByPosteriorProbability / ...IgnoringGaps (kind = SCORE_*, impl/pairwiseAligner.c:1562-1597)
        of every pair's alignment -> float64[n]"""
        out = np.zeros(max(self.n, 1), dtype=np.float64)
        _check(lib.cpb_batch_score_alignments(self.h, int(kind), C.c_void_p(out.ctypes.data)))
        return out[: self.n]

    def alignment_cigars(self):
        """-> (offsets[n+1] int64, ops[count, 2] int32 (type OP_*, length)): the cigar operations cPecanRealign writes for every pair's
        alignment, built on the device from the alignment list"""
        off = np.zeros(self.n + 1, dtype=np.int64)
        _check(lib.cpb_batch_alignment_cigars(self.h, C.c_void_p(off.ctypes.data)))
        m = int(off[-1])
        ops = np.zeros((max(m, 1), 2), dtype=np.int32)
        _check(lib.cpb_batch_fetch_cigars(self.h, C.c_void_p(ops.ctypes.data)))
        return off, ops[:m]

    def alignments_from_cigars(self, cigars, trim=0):
        """replaces the alignment list with every MATCH column at [trim, L - trim) of every pair's cigar (offsets[n+1], ops[m, 2] as
        alignment_cigars returns them), x ascending, each weighed with its weight in list 0 of the last run (0 if it is not there): what
        cPecanRealign --rescoreOriginalAlignment scores"""
        oo, ops = _cigar_arrays(cigars)
        _check(lib.cpb_batch_alignments_from_cigars(self.h, _ptr(oo), _ptr(ops) if len(ops) else None, int(trim)))

    def anchors_from_alignments(self, params):
        """replaces every pair's anchors with those its alignment gives (params.constraintDiagonalTrim, params.diagonalExpansion): the
        anchors cPecanRealign's job_prepare builds from the cigar of that alignment; the next run plans anew with them"""
        _check(lib.cpb_batch_anchors_from_alignments(self.h, C.byref(params) if params is not None else None))

    def fetch_expectations(self, per_pair=True):
        L = hmm_len(self.S)
        pp = np.zeros((self.n, L), dtype=np.float64) if per_pair else None
        tot = np.zeros(L, dtype=np.float64)
        _check(lib.cpb_batch_fetch_expectations(self.h, C.c_void_p(pp.ctypes.data) if pp is not None and self.n else None,
                                                C.c_void_p(tot.ctypes.data)))
        return pp, tot

    def device_expectation_total_ptr(self):
        return lib.cpb_batch_device_expectation_total(self.h)

    def fetch_forward(self):
        out = np.zeros(max(self.n, 1), dtype=np.float64)
        _check(lib.cpb_batch_fetch_forward(self.h, C.c_void_p(out.ctypes.data)))
        return out[: self.n]

    def close(self):
        if self.h:
            # cpb_batch_destroy reads the batch's context (device, buffer pools): after the context is closed it must not run; the batch's
            # device memory then goes back with the process
            if self.ctx.h:
                lib.cpb_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- the reference's one-pair-per-call functions, on top of a 1-element batch ----
def _one(sM, sX, sY, anchorPairs, p, raggedLeft, raggedRight, mode, ctx=None):
    ctx = ctx or default_context()
    b = Batch(ctx, [sX], [sY], [anchorPairs], [int(raggedLeft)], [int(raggedRight)])
    b.run(sM, p, mode)
    return b


def getAlignedPairsUsingAnchors(sM, sX, sY, anchorPairs, p, alignmentHasRaggedLeftEnd=False, alignmentHasRaggedRightEnd=False, ctx=None):
    """-> list of (pInt, x, y) (inc/pairwiseAligner.h:75)"""
    b = _one(sM, sX, sY, anchorPairs, p, alignmentHasRaggedLeftEnd, alignmentHasRaggedRightEnd, MODE_ALIGNED_PAIRS, ctx)
    _, tri = b.fetch_pairs(0)
    b.close()
    return [tuple(int(v) for v in t) for t in tri]


def getAlignedPairsWithIndelsUsingAnchors(sM, sX, sY, anchorPairs, p, alignmentHasRaggedLeftEnd=False, alignmentHasRaggedRightEnd=False, ctx=None):
    """-> (alignedPairs, gapXPairs, gapYPairs) (inc/pairwiseAligner.h:77)"""
    b = _one(sM, sX, sY, anchorPairs, p, alignmentHasRaggedLeftEnd, alignmentHasRaggedRightEnd, MODE_ALIGNED_PAIRS_INDELS, ctx)
    out = []
    for which in range(3):
        _, tri = b.fetch_pairs(which)
        out.append([tuple(int(v) for v in t) for t in tri])
    b.close()
    return tuple(out)


def getExpectationsUsingAnchors(sM, hmmExpectations, sX, sY, anchorPairs, p, alignmentHasRaggedLeftEnd=False, alignmentHasRaggedRightEnd=False, ctx=None):
    """Accumulates into hmmExpectations (a float64 array of hmm_len(S): transitions, emissions, likelihood) (inc/pairwiseAligner.h:105)."""
    b = _one(sM, sX, sY, anchorPairs, p, alignmentHasRaggedLeftEnd, alignmentHasRaggedRightEnd, MODE_EXPECTATIONS, ctx)
    _, tot = b.fetch_expectations(per_pair=False)
    b.close()
    hmmExpectations += tot
    return hmmExpectations


# ---- the same from raw sequences, anchored on the device as the reference's getAlignedPairs anchors them ----
def _one_anchored(sM, sX, sY, p, raggedLeft, raggedRight, mode, ctx):
    b = Batch.anchored(ctx or default_context(), [sX], [sY], p, [int(raggedLeft)], [int(raggedRight)])
    b.run(sM, p, mode)
    return b


def getAlignedPairs(sM, sX, sY, p, alignmentHasRaggedLeftEnd=False, alignmentHasRaggedRightEnd=False, ctx=None):
    """-> list of (pInt, x, y) (inc/pairwiseAligner.h:58)"""
    b = _one_anchored(sM, sX, sY, p, alignmentHasRaggedLeftEnd, alignmentHasRaggedRightEnd, MODE_ALIGNED_PAIRS, ctx)
    _, tri = b.fetch_pairs(0)
    b.close()
    return [tuple(int(v) for v in t) for t in tri]


def getAlignedPairsWithIndels(sM, sX, sY, p, alignmentHasRaggedLeftEnd=False, alignmentHasRaggedRightEnd=False, ctx=None):
    """-> (alignedPairs, gapXPairs, gapYPairs) (inc/pairwiseAligner.h:60)"""
    b = _one_anchored(sM, sX, sY, p, alignmentHasRaggedLeftEnd, alignmentHasRaggedRightEnd, MODE_ALIGNED_PAIRS_INDELS, ctx)
    out = []
    for which in range(3):
        _, tri = b.fetch_pairs(which)
        out.append([tuple(int(v) for v in t) for t in tri])
    b.close()
    return tuple(out)


def getExpectations(sM, hmmExpectations, sX, sY, p, alignmentHasRaggedLeftEnd=False, alignmentHasRaggedRightEnd=False, ctx=None):
    """Accumulates into hmmExpectations, as getExpectationsUsingAnchors (inc/pairwiseAligner.h:74)."""
    b = _one_anchored(sM, sX, sY, p, alignmentHasRaggedLeftEnd, alignmentHasRaggedRightEnd, MODE_EXPECTATIONS, ctx)
    _, tot = b.fetch_expectations(per_pair=False)
    b.close()
    hmmExpectations += tot
    return hmmExpectations


def getShiftedMEAAlignment(seqX, seqY, anchorPairs, p, sM, alignmentHasRaggedLeftEnd=False, alignmentHasRaggedRightEnd=False, ctx=None):
    """-> (list of (pInt, x, y), alignmentScore) (impl/pairwiseAligner.c:1769-1792): one ALIGNED_PAIRS_INDELS run, then the maximal expected
    accuracy alignment with p.gapGamma and its left shift, on the device"""
    b = _one(sM, seqX, seqY, anchorPairs, p, alignmentHasRaggedLeftEnd, alignmentHasRaggedRightEnd, MODE_ALIGNED_PAIRS_INDELS, ctx)
    try:
        score = float(b.mea(p.gapGamma, left_shift=True)[0])
        _, tri = b.fetch_alignments()
    finally:
        b.close()
    return [tuple(int(v) for v in t) for t in tri], score


def computeForwardProbability(seqX, seqY, anchorPairs, p, sM, alignmentHasRaggedLeftEnd=False, alignmentHasRaggedRightEnd=False, ctx=None):
    """inc/pairwiseAligner.h:56"""
    b = _one(sM, seqX, seqY, anchorPairs, p, alignmentHasRaggedLeftEnd, alignmentHasRaggedRightEnd, MODE_FORWARD, ctx)
    v = float(b.fetch_forward()[0])
    b.close()
    return v
