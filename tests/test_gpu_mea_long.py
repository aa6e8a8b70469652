"""The MEA of long pairs on the device and in batches: cpb_batch_mea, with its walk-back skipping chunks and 1024-triple blocks of the
reference-ordered list that hold no predecessor (decode_kernels.cuh, k_mea_summaries / k_mea), against libcpecan.so's host function on
the lists in the reference's order, and getShiftedMEAAlignmentBatch of libcpecan.so against per-pair getShiftedMEAAlignment.  Pairs of
1 kb to 100 kb with many traceback blocks and split regions.  Every comparison is exact: the same triples in the same order and the same
bits of alignmentScore."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

if __name__ == "__main__":  # the worker of test_batch_over_two_contexts_of_one_gpu, run as a script
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import cpecan_b200 as cp  # noqa: E402
import helpers  # noqa: E402
from cpecan_b200 import synth  # noqa: E402
from host_anchors import HostAnchorer  # noqa: E402
from test_gpu_alignments import PAIRS, SlabHost, _per_pair, _same_bits  # noqa: E402

pytestmark = pytest.mark.gpu

HOST_SO = os.path.join(helpers.ROOT, "cpecan_b200", "lib", "libcpecan.so")


def long_pairs():
    """(name, sX, sY, raggedLeft, raggedRight): evolved pairs of 1 kb to 100 kb"""
    out = []
    for length, n in ((1000, 3), (10000, 3), (40000, 2), (100000, 2)):
        packed = synth.evolved_pairs(n, length, seed=700 + length // 1000, trim=0, expansion=0)
        out += [("evolved%d_%d" % (length, i),) + tuple(synth.unpack(packed, i)[:2]) + (i == 1, i == 2) for i in range(n)]
    return out


LONG = long_pairs()


def param_sets():
    defaults = cp.pairwiseAlignmentBandingParameters_construct()
    split = cp.pairwiseAlignmentBandingParameters_construct()  # regions split at every anchor gap above a small matrix
    split.splitMatrixBiggerThanThis = 2000
    split.minDiagsBetweenTraceBack = 300  # shorter traceback blocks: more of them per region
    return {"defaults": defaults, "split": split}


@pytest.fixture(scope="module")
def host():
    return SlabHost()


def _batch(ctx, p, pairs=LONG):
    return cp.Batch.anchored(ctx, [q[1] for q in pairs], [q[2] for q in pairs], p, [q[3] for q in pairs], [q[4] for q in pairs])


def _device_mea(b, gamma):
    out = {}
    for shift in (False, True):
        scores = b.mea(gamma, left_shift=shift)
        out[shift] = (_per_pair(*b.fetch_alignments()), scores)
    return out


@pytest.mark.parametrize("which", ["defaults", "split"])
def test_long_mea_equals_the_host(ctx, host, which):
    p = param_sets()[which]
    b = _batch(ctx, p)
    try:
        b.run(cp.stateMachine5_construct(), p, cp.MODE_ALIGNED_PAIRS_INDELS)
        st = b.stats()
        if which == "defaults":
            assert st.nBlocks > 4 * st.nRegions  # many traceback blocks per region: the reference order puts the later ones first
        else:
            assert st.nRegions > 2 * len(LONG) and st.nBlocks > st.nRegions
        l0, l1, l2 = (_per_pair(*b.fetch_pairs(k, reference_order=True)) for k in range(3))
        assert max(len(l) for l in l0) > 2 * 32768  # lists longer than a group of 32 summary blocks of 1024 triples
        for gamma in sorted({float(p.gapGamma), 0.0}):
            got = _device_mea(b, gamma)
            for i, q in enumerate(LONG):
                want, score = host.mea(l0[i], l1[i], l2[i], len(q[1]), len(q[2]), gamma)
                assert np.array_equal(got[False][0][i], want), "%s, gapGamma %g, %s: MEA differs" % (which, gamma, q[0])
                assert _same_bits(got[False][1][i], score), "%s, gapGamma %g, %s: alignmentScore %r, host %r" % (which, gamma, q[0], got[False][1][i], score)
                assert _same_bits(got[True][1][i], score)
                shifted = host.left_shift(want, q[1].decode(), q[2].decode())
                assert np.array_equal(got[True][0][i], shifted), "%s, gapGamma %g, %s: left shift differs" % (which, gamma, q[0])
    finally:
        b.close()


def test_small_scratch_budget_gives_the_same_long_mea(ctx):
    """a budget that holds the work arrays of one or two 100 kb pairs at a time: many chunks of pairs"""
    p = param_sets()["split"]
    b = _batch(ctx, p)
    try:
        b.run(cp.stateMachine5_construct(), p, cp.MODE_ALIGNED_PAIRS_INDELS)
        want = _device_mea(b, float(p.gapGamma))
        ctx.set_scratch_budget(12 << 20)
        got = _device_mea(b, float(p.gapGamma))
        for shift in (False, True):
            assert all(np.array_equal(g, w) for g, w in zip(got[shift][0], want[shift][0]))
            assert _same_bits(got[shift][1], want[shift][1])
        ctx.set_scratch_budget(1 << 20)  # less than one 100 kb pair needs
        with pytest.raises(cp.CpbError, match="error 5"):
            b.mea(float(p.gapGamma))
    finally:
        ctx.set_scratch_budget(0)
        b.close()


# ---- getShiftedMEAAlignmentBatch of libcpecan.so ----

class Lib:
    """ctypes mirror of the entry points of libcpecan.so this file calls"""

    def __init__(self):
        L = self.L = C.CDLL(HOST_SO)
        vp, i64 = C.c_void_p, C.c_int64
        for f in ("stateMachine5_construct", "pairwiseAlignmentBandingParameters_construct", "getShiftedMEAAlignment", "getShiftedMEAAlignmentBatch"):
            getattr(L, f).restype = vp
        L.stateMachine5_construct.argtypes = [C.c_int]
        L.getShiftedMEAAlignment.argtypes = [C.c_char_p, C.c_char_p, vp, vp, vp, C.c_bool, C.c_bool, C.POINTER(C.c_double)]
        L.getShiftedMEAAlignmentBatch.argtypes = [vp, i64, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.POINTER(vp), vp, vp, vp, vp]
        self.free = C.CDLL(None).free
        self.free.argtypes = [vp]
        self.h = SlabHost()

    def per_pair(self, sM, p, sx, sy, anchors, rl, rr):
        score = C.c_double()
        a = self.h.to_list(anchors)
        out = self.h.from_list(self.L.getShiftedMEAAlignment(sx, sy, a, p, sM, rl, rr, C.byref(score)))
        self.h.L.stList_destruct(a)
        return out, score.value

    def batch(self, sM, p, sxs, sys_, anchors, rl=None, rr=None, want_scores=True):
        n = len(sxs)
        lists = [self.h.to_list(a) for a in anchors]
        arr = (C.c_void_p * max(n, 1))(*lists)
        bools = lambda v: None if v is None else C.cast((C.c_bool * max(n, 1))(*[bool(x) for x in v]), C.c_void_p)  # noqa: E731
        scores = np.full(max(n, 1), np.nan)
        res = self.L.getShiftedMEAAlignmentBatch(sM, n, (C.c_char_p * max(n, 1))(*sxs), (C.c_char_p * max(n, 1))(*sys_), arr, p, bools(rl), bools(rr),
                                                 C.c_void_p(scores.ctypes.data) if want_scores else None)
        got = C.cast(res, C.POINTER(C.c_void_p))
        out = [self.h.from_list(got[i]) for i in range(n)]
        self.free(res)
        for a in lists:
            self.h.L.stList_destruct(a)
        return out, scores[:n]


def batch_problems():
    names = ("evolved1000_0", "evolved12000_1", "tandem", "iupac", "ragged", "empty_x", "one_base", "n_runs")
    return [q for q in PAIRS if q[0] in names] + LONG[:4] + [LONG[-1]]


def check_batch_against_per_pair():
    """getShiftedMEAAlignmentBatch with ragged ends, with NULL ragged arrays and with a NULL score array, against getShiftedMEAAlignment
    per problem; raises AssertionError on the first difference"""
    lib = Lib()
    sM, p = lib.L.stateMachine5_construct(0), lib.L.pairwiseAlignmentBandingParameters_construct()
    ha = HostAnchorer()
    hp = ha.params(cp.pairwiseAlignmentBandingParameters_construct())
    probs = batch_problems()
    sxs, sys_ = [q[1] for q in probs], [q[2] for q in probs]
    anchors = [ha.anchors(q[1], q[2], hp) for q in probs]
    rl, rr = [bool(q[3]) for q in probs], [bool(q[4]) for q in probs]
    for ragged in (True, False):
        got, scores = lib.batch(sM, p, sxs, sys_, anchors, rl if ragged else None, rr if ragged else None)
        for i, q in enumerate(probs):
            want, score = lib.per_pair(sM, p, q[1], q[2], anchors[i], rl[i] and ragged, rr[i] and ragged)
            assert np.array_equal(got[i], want), "%s (ragged %s): triples differ" % (q[0], ragged)
            assert _same_bits(scores[i], score), "%s (ragged %s): alignmentScore %r, per pair %r" % (q[0], ragged, scores[i], score)
    again, _ = lib.batch(sM, p, sxs, sys_, anchors, rl, rr, want_scores=False)
    first, _ = lib.batch(sM, p, sxs, sys_, anchors, rl, rr)
    assert all(np.array_equal(a, b) for a, b in zip(again, first))
    assert lib.batch(sM, p, [], [], [])[0] == []


def _run_worker(devices):
    env = dict(os.environ)
    env.pop("CPECAN_DEVICES", None)
    env.pop("CPECAN_DEVICE", None)
    env["CPECAN_DEVICE_LIST"] = devices
    out = subprocess.run([sys.executable, os.path.abspath(__file__)], capture_output=True, text=True, env=env)
    assert out.returncode == 0 and "batch ok" in out.stdout, out.stdout + out.stderr


def test_batch_equals_per_pair():
    _run_worker("0")


def test_batch_over_two_contexts_of_one_gpu():
    """CPECAN_DEVICE_LIST=0,0: the problems are dealt over two contexts (one host thread and stream each) of the same GPU"""
    _run_worker("0,0")


if __name__ == "__main__":
    check_batch_against_per_pair()
    print("batch ok")
