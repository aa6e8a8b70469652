"""Alignments decoded on the device (cpb_batch_ordered_chain, cpb_batch_mea, cpb_batch_score_alignments; decode_kernels.cuh) against the
host functions of libcpecan.so (host/realign.c) run in the same process on the lists the device hands over: the same triples in the same
order, the same double bits.  Every comparison is exact."""
import ctypes as C
import os

import numpy as np
import pytest

import cpecan_b200 as cp
import helpers
from cpecan_b200 import synth
from host_anchors import HostAnchorer
from test_realign_host import Host, Ref

pytestmark = pytest.mark.gpu


class SlabHost(Host):
    """Host, with input lists cut from one slab (cpecan_tripleList_construct) instead of one ctypes call per tuple"""

    def __init__(self):
        super().__init__()
        self.L.cpecan_tripleList_construct.restype = C.c_void_p
        self.L.cpecan_tripleList_construct.argtypes = [C.c_void_p, C.c_int64]

    def to_list(self, triples):
        t = np.ascontiguousarray(np.asarray(triples).reshape(-1, 3), dtype=np.int32)
        keep = t if len(t) else np.zeros((1, 3), dtype=np.int32)
        return self.L.cpecan_tripleList_construct(keep.ctypes.data, len(t))


@pytest.fixture(scope="module")
def host():
    return SlabHost()


def _rs(rng, n):
    return synth.random_sequence(rng, n, acgt_only=True).encode()


def _mutate(rng, s, rate):
    a = bytearray(s)
    for i in np.nonzero(rng.random(len(a)) < rate)[0]:
        a[i] = b"ACGT"[(b"ACGT".index(a[i]) + int(rng.integers(1, 4))) % 4]
    return bytes(a)


def mixed_pairs():
    """(name, sX, sY, raggedLeft, raggedRight)"""
    rng = np.random.default_rng(4242)
    out = []
    for length, n in ((400, 2), (1000, 2), (3000, 1), (12000, 2)):
        packed = synth.evolved_pairs(n, length, seed=90 + length, trim=0, expansion=0)
        out += [("evolved%d_%d" % (length, i),) + tuple(synth.unpack(packed, i)[:2]) + (i % 2, 0) for i in range(n)]
    s = _rs(rng, 1500)
    out.append(("identical", s, s, 0, 0))
    unit = _rs(rng, 23)
    tandem = unit * 60
    out.append(("tandem", tandem, _mutate(rng, tandem, 0.03), 0, 1))
    out.append(("tandem_same", unit * 40, unit * 40, 0, 0))
    out.append(("unrelated", _rs(rng, 800), _rs(rng, 800), 0, 0))
    t = _rs(rng, 2000)
    u = _mutate(rng, t, 0.04)
    out.append(("lower", t[:700].lower() + t[700:], u[:300] + u[300:1200].lower() + u[1200:], 0, 0))
    out.append(("n_runs", t[:500] + b"N" * 80 + t[580:], u[:500] + b"n" * 80 + u[580:], 1, 1))
    out.append(("iupac", t[:900] + b"xyzN" * 20 + t[980:], u[:900] + b"xyzN" * 20 + u[980:], 0, 0))
    out.append(("iupac_mixed", t[:1000] + b"RYKM" * 10 + t[1040:], u[:1000] + b"RRYY" * 10 + u[1040:], 0, 0))
    out.append(("ragged", t[200:1600], u, 1, 1))
    out.append(("empty_x", b"", _rs(rng, 300), 0, 0))
    out.append(("empty_y", _rs(rng, 300), b"", 0, 0))
    out.append(("empty_both", b"", b"", 0, 0))
    out.append(("one_base", b"A", b"A", 0, 0))
    out.append(("one_base_vs", b"c", _rs(rng, 40), 0, 0))
    return out


PAIRS = mixed_pairs()


def param_sets():
    defaults = cp.pairwiseAlignmentBandingParameters_construct()
    realign = cp.pairwiseAlignmentBandingParameters_construct()  # cPecanRealign's (host/cPecanRealign.c:284-289)
    realign.constraintDiagonalTrim, realign.splitMatrixBiggerThanThis, realign.diagonalExpansion = 0, 10, 4
    em = cp.pairwiseAlignmentBandingParameters_construct()  # cPecanEm's (host/cPecanEm.c:146-148)
    em.constraintDiagonalTrim, em.diagonalExpansion, em.splitMatrixBiggerThanThis = 0, 10, 3000 * 3000
    return {"defaults": defaults, "realign": realign, "em": em}


def _model(S):
    return cp.stateMachine5_construct() if S == 5 else cp.stateMachine3_construct()


def _batch(ctx, anchoring, p, pairs=PAIRS):
    sx, sy = [q[1] for q in pairs], [q[2] for q in pairs]
    rl, rr = [q[3] for q in pairs], [q[4] for q in pairs]
    if anchoring == "device":
        return cp.Batch.anchored(ctx, sx, sy, p, rl, rr)
    ha = HostAnchorer()
    hp = ha.params(p)
    return cp.Batch(ctx, sx, sy, [ha.anchors(x, y, hp) for x, y in zip(sx, sy)], rl, rr)


def _per_pair(off, tri):
    return [tri[off[i]:off[i + 1]].astype(np.int64) for i in range(len(off) - 1)]


def _same_bits(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return bool(np.all((a.view(np.int64) == b.view(np.int64)) | (np.isnan(a) & np.isnan(b))))


def _check_scores(host, b, pairs, alns, what):
    want = np.array([host.scores(q[1].decode(), q[2].decode(), a) for q, a in zip(pairs, alns)], dtype=np.float64).reshape(-1, 4)
    for kind in range(4):
        got = b.score_alignments(kind)
        assert _same_bits(got, want[:, kind]), "%s: score kind %d differs: %s" % (what, kind, [(q[0], g, w) for q, g, w in zip(pairs, got, want[:, kind])
                                                                                           if not _same_bits(g, w)][:5])
    empty = [i for i, a in enumerate(alns) if len(a) == 0]
    if empty:
        assert np.all(np.isnan(b.score_alignments(cp.SCORE_IDENTITY_IGNORING_GAPS)[empty]))


def _check_chains(host, b, pairs, what):
    lists = _per_pair(*b.fetch_pairs(0))
    for gamma in (0.0, 0.5, 0.85, 1.0):
        b.ordered_chain(gamma)
        got = _per_pair(*b.fetch_alignments())
        for q, l0, g in zip(pairs, lists, got):
            want = host.chain(l0, q[1].decode(), q[2].decode(), gamma)
            assert np.array_equal(g, want), "%s, matchGamma %g, %s: %d device pairs, %d host pairs" % (what, gamma, q[0], len(g), len(want))
        if gamma == 0.85:
            _check_scores(host, b, pairs, got, what + " chain")
    return lists


SETUPS = [(S, which, "device") for S in (5, 3) for which in ("defaults", "realign", "em")] + [(5, "defaults", "caller")]


@pytest.mark.parametrize("S,which,anchoring", SETUPS)
def test_decoders_equal_the_hosts(ctx, host, S, which, anchoring):
    p = param_sets()[which]
    sM = _model(S)
    b = _batch(ctx, anchoring, p)
    what = "%d-state, %s parameters, %s anchors" % (S, which, anchoring)
    # chain, on the posteriors and on the reweighted posteriors
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)
    assert sum(1 for l0 in _per_pair(*b.fetch_pairs(0)) if len(l0) == 0) >= 3  # the empty inputs give empty lists
    _check_chains(host, b, PAIRS, what)
    b.reweight_pairs(p.gapGamma)
    _check_chains(host, b, PAIRS, what + ", reweighted")
    # MEA and its left shift on the lists in the reference's order
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS_INDELS)
    st = b.stats()
    if which == "defaults":
        assert st.nBlocks > st.nRegions  # some pairs have several traceback blocks: list order matters
    l0, l1, l2 = (_per_pair(*b.fetch_pairs(k, reference_order=True)) for k in range(3))
    for gamma in sorted({float(p.gapGamma), 0.0, 0.9}):
        scores = b.mea(gamma, left_shift=False)
        got = _per_pair(*b.fetch_alignments())
        meas = []
        for i, q in enumerate(PAIRS):
            want, score = host.mea(l0[i], l1[i], l2[i], len(q[1]), len(q[2]), gamma)
            meas.append(want)
            assert np.array_equal(got[i], want), "%s, gapGamma %g, %s: MEA differs" % (what, gamma, q[0])
            assert _same_bits(scores[i], score), "%s, gapGamma %g, %s: alignmentScore %r, host %r" % (what, gamma, q[0], scores[i], score)
        _check_scores(host, b, PAIRS, got, what + " MEA")
        shifted_scores = b.mea(gamma, left_shift=True)
        assert _same_bits(shifted_scores, scores)
        got = _per_pair(*b.fetch_alignments())
        for i, q in enumerate(PAIRS):
            want = host.left_shift(meas[i], q[1].decode(), q[2].decode())
            assert np.array_equal(got[i], want), "%s, gapGamma %g, %s: left shift differs" % (what, gamma, q[0])
        _check_scores(host, b, PAIRS, got, what + " shifted MEA")
    b.close()


def test_mea_equals_the_reference_build(ctx, host):
    """the device MEA on multi-block lists against the reference's own getMaximalExpectedAccuracyPairwiseAlignment (oracle/_ref)"""
    ref = helpers.ref_oracle()
    if ref is None:
        pytest.skip("oracle/_ref not built here")
    ref = Ref(ref)
    p = param_sets()["defaults"]
    b = _batch(ctx, "device", p)
    b.run(_model(5), p, cp.MODE_ALIGNED_PAIRS_INDELS)
    l0, l1, l2 = (_per_pair(*b.fetch_pairs(k, reference_order=True)) for k in range(3))
    scores = b.mea(p.gapGamma, left_shift=False)
    got = _per_pair(*b.fetch_alignments())
    for i, q in enumerate(PAIRS):
        want, score = ref.mea(l0[i], l1[i], l2[i], len(q[1]), len(q[2]), float(p.gapGamma))
        assert np.array_equal(got[i], want) and _same_bits(scores[i], score), q[0]
    b.close()


def test_shifted_mea_equals_libcpecan(ctx):
    """end to end: getShiftedMEAAlignment of libcpecan.so (host MEA and left shift) against the device's, on the same anchors"""
    L = C.CDLL(os.path.join(helpers.ROOT, "cpecan_b200", "lib", "libcpecan.so"))
    vp = C.c_void_p
    for f in ("stateMachine5_construct", "pairwiseAlignmentBandingParameters_construct", "getShiftedMEAAlignment"):
        getattr(L, f).restype = vp
    L.getShiftedMEAAlignment.argtypes = [C.c_char_p, C.c_char_p, vp, vp, vp, C.c_bool, C.c_bool, C.POINTER(C.c_double)]
    h = SlabHost()
    hsM = L.stateMachine5_construct(0)
    hp = L.pairwiseAlignmentBandingParameters_construct()
    p = cp.pairwiseAlignmentBandingParameters_construct()
    ha = HostAnchorer()
    names = ("evolved1000_0", "evolved12000_1", "tandem", "iupac", "ragged", "empty_x", "one_base")
    for q in [q for q in PAIRS if q[0] in names]:
        anchors = ha.anchors(q[1], q[2], ha.params(p))
        score = C.c_double()
        want = h.from_list(L.getShiftedMEAAlignment(q[1], q[2], h.to_list(anchors), hp, hsM, bool(q[3]), bool(q[4]), C.byref(score)))
        got, dscore = cp.getShiftedMEAAlignment(q[1], q[2], anchors, p, _model(5), bool(q[3]), bool(q[4]), ctx=ctx)
        assert np.array_equal(np.array(got, dtype=np.int64).reshape(-1, 3), want), q[0]
        assert _same_bits(dscore, score.value), q[0]


def test_small_scratch_budget_gives_the_same_alignments(ctx):
    p = param_sets()["defaults"]
    b = _batch(ctx, "device", p)
    sM = _model(5)
    want = {}
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS_INDELS)
    try:
        for budget in (0, 1 << 20):
            ctx.set_scratch_budget(budget)
            b.ordered_chain(0.5)
            chain = b.fetch_alignments()
            scores = b.mea(p.gapGamma)
            mea = b.fetch_alignments()
            if budget == 0:
                want = (chain, scores, mea)
            else:
                for g, w in zip((chain[0], chain[1], mea[0], mea[1]), (want[0][0], want[0][1], want[2][0], want[2][1])):
                    assert np.array_equal(g, w)
                assert _same_bits(scores, want[1])
        ctx.set_scratch_budget(8192)  # less than a 12 kb pair's work arrays
        for call in (lambda: b.ordered_chain(0.5), lambda: b.mea(p.gapGamma)):
            with pytest.raises(cp.CpbError, match="error 5"):
                call()
    finally:
        ctx.set_scratch_budget(0)
    b.close()


def test_error_paths(ctx):
    p = param_sets()["defaults"]
    pairs = [q for q in PAIRS if q[0] in ("evolved1000_0", "tandem", "empty_y")]
    b = _batch(ctx, "device", p, pairs)
    sM = _model(5)

    def refused(call, name):
        with pytest.raises(cp.CpbError, match="error 2: %s" % name):
            call()

    refused(lambda: b.fetch_alignments(), "cpb_batch_fetch_alignments")  # nothing decoded yet
    refused(lambda: b.ordered_chain(0.5), "cpb_batch_ordered_chain")    # nothing run yet
    for mode in (cp.MODE_EXPECTATIONS, cp.MODE_FORWARD):
        b.run(sM, p, mode)
        refused(lambda: b.ordered_chain(0.5), "cpb_batch_ordered_chain")
        refused(lambda: b.mea(0.5), "cpb_batch_mea")
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)
    refused(lambda: b.mea(0.5), "cpb_batch_mea")  # no gap lists
    refused(lambda: b.score_alignments(cp.SCORE_IDENTITY), "cpb_batch_score_alignments")
    for g in (-0.1, 1.5, float("nan")):
        refused(lambda: b.ordered_chain(g), "cpb_batch_ordered_chain")
    b.ordered_chain(0.85)
    off, tri = b.fetch_alignments()
    assert off[-1] > 0 and int(cp.lib.cpb_batch_alignments_count(b.h)) == off[-1]
    for kind in (-1, 4):
        refused(lambda: b.score_alignments(kind), "cpb_batch_score_alignments")
    b.reweight_pairs(0.5)  # does not touch the alignment list
    off2, tri2 = b.fetch_alignments()
    assert np.array_equal(off, off2) and np.array_equal(tri, tri2)
    refused(lambda: b.mea(0.5), "cpb_batch_mea")  # a refused decode leaves no list, whatever the reason
    refused(lambda: b.fetch_alignments(), "cpb_batch_fetch_alignments")
    b.ordered_chain(0.85)
    refused(lambda: b.ordered_chain(2.0), "cpb_batch_ordered_chain")
    refused(lambda: b.fetch_alignments(), "cpb_batch_fetch_alignments")
    b.ordered_chain(0.85)
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS_INDELS)  # a run clears it
    assert int(cp.lib.cpb_batch_alignments_count(b.h)) == 0
    refused(lambda: b.fetch_alignments(), "cpb_batch_fetch_alignments")
    for g in (-1.0, float("inf"), float("nan")):
        refused(lambda: b.mea(g), "cpb_batch_mea")
    refused(lambda: b.fetch_alignments(), "cpb_batch_fetch_alignments")  # a refused decode leaves no list
    b.mea(0.5)
    assert b.fetch_alignments()[0][-1] > 0
    b.close()


@pytest.mark.parametrize("which", ["defaults", "realign"])
def test_device_reference_order_equals_the_hosts(ctx, which):
    """the permutation k_ref_order makes on the device (what cpb_batch_mea walks) against cpb_batch_fetch_pairs_reference_order, triple
    for triple, in both aligned-pair modes and under a scratch budget that forces many chunks"""
    lib = cp.lib
    lib.cpb_debug_reference_order.argtypes = [C.c_void_p]
    p = param_sets()[which]
    b = _batch(ctx, "device", p)
    try:
        for mode in (cp.MODE_ALIGNED_PAIRS_INDELS, cp.MODE_ALIGNED_PAIRS):
            b.run(_model(5), p, mode)
            if which == "defaults":
                st = b.stats()
                assert st.nBlocks > st.nRegions
            want_off, want = b.fetch_pairs(0, reference_order=True)
            _, device_order = b.fetch_pairs(0)
            assert not np.array_equal(want, device_order) or which != "defaults"  # the permutation is not the identity
            for budget in (0, 1 << 20):
                ctx.set_scratch_budget(budget)
                assert lib.cpb_debug_reference_order(b.h) == 0, lib.cpb_last_error()
                off, got = b.fetch_alignments()
                assert np.array_equal(off, want_off) and np.array_equal(got, want)
    finally:
        ctx.set_scratch_budget(0)
        b.close()
