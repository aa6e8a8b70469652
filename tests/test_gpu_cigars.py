"""Cigar operations built on the device from the alignment list (cpb_batch_alignment_cigars, cpb_batch_fetch_cigars; k_cigar_count and
k_cigar_write of decode_kernels.cuh) against ops_from_columns, the Python statement of cPecanRealign's pairs_to_alignment, applied to the
fetched alignment.  Every comparison is exact."""
import ctypes as C

import numpy as np
import pytest

import cpecan_b200 as cp
from test_gpu_alignments import PAIRS, _batch, _model, param_sets
from test_gpu_realign_cli import ops_from_columns

pytestmark = pytest.mark.gpu


def _check_cigars(b, pairs, what):
    aoff, tri = b.fetch_alignments()
    off, ops = b.alignment_cigars()
    assert off.shape == (len(pairs) + 1,) and off[0] == 0 and ops.shape == (off[-1], 2)
    for i, q in enumerate(pairs):
        cols = [(int(t[1]), int(t[2])) for t in tri[aoff[i]:aoff[i + 1]]]
        want = ops_from_columns(cols, len(q[1]), len(q[2]))
        got = [(int(t), int(n)) for t, n in ops[off[i]:off[i + 1]]]
        assert got == want, "%s, %s: device %s..., host %s..." % (what, q[0], got[:6], want[:6])
        assert len(got) <= 3 * len(cols) + 2
    return off, ops


@pytest.mark.parametrize("S,which", [(S, which) for S in (5, 3) for which in ("defaults", "realign")])
def test_cigars_equal_the_columns(ctx, S, which):
    p = param_sets()[which]
    sM = _model(S)
    b = _batch(ctx, "device", p)
    what = "%d-state, %s parameters" % (S, which)
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)
    for reweighted in (False, True):
        if reweighted:
            b.reweight_pairs(p.gapGamma)
        for gamma in (0.0, 0.5, 0.85, 1.0):
            b.ordered_chain(gamma)
            off, ops = _check_cigars(b, PAIRS, "%s, chain at %g%s" % (what, gamma, ", reweighted" if reweighted else ""))
            if gamma == 0.85:
                kinds = set(ops[:, 0].tolist())
                assert kinds == {cp.OP_MATCH, cp.OP_INDEL_X, cp.OP_INDEL_Y}
                # the empty sequences: [INDEL_Y 300], [INDEL_X 300], nothing
                for name, want in (("empty_x", [(cp.OP_INDEL_Y, 300)]), ("empty_y", [(cp.OP_INDEL_X, 300)]), ("empty_both", [])):
                    i = [q[0] for q in PAIRS].index(name)
                    assert [tuple(o) for o in ops[off[i]:off[i + 1]].tolist()] == want
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS_INDELS)
    for shift in (False, True):
        b.mea(p.gapGamma, left_shift=shift)
        _check_cigars(b, PAIRS, "%s, MEA%s" % (what, " shifted" if shift else ""))
    b.close()


def test_small_scratch_budget_gives_the_same_cigars(ctx):
    p = param_sets()["defaults"]
    b = _batch(ctx, "device", p)
    b.run(_model(5), p, cp.MODE_ALIGNED_PAIRS)
    b.ordered_chain(0.5)
    want = _check_cigars(b, PAIRS, "budget 0")
    try:
        ctx.set_scratch_budget(1 << 20)  # the chain runs in many chunks
        b.ordered_chain(0.5)
        got = _check_cigars(b, PAIRS, "budget 1 MB")
    finally:
        ctx.set_scratch_budget(0)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    b.close()


def test_error_paths(ctx):
    lib = cp.lib
    p = param_sets()["defaults"]
    pairs = [q for q in PAIRS if q[0] in ("evolved1000_0", "tandem", "empty_y")]
    b = _batch(ctx, "device", p, pairs)
    sM = _model(5)
    off = np.zeros(len(pairs) + 1, dtype=np.int64)
    buf = np.zeros((1 << 16, 2), dtype=np.int32)

    def refused(call, name):
        with pytest.raises(cp.CpbError, match="error 2: %s" % name):
            call()

    build = lambda: b.alignment_cigars()  # noqa: E731
    fetch = lambda: cp.binding._check(lib.cpb_batch_fetch_cigars(b.h, C.c_void_p(buf.ctypes.data)))  # noqa: E731
    refused(build, "cpb_batch_alignment_cigars")  # nothing decoded yet
    refused(fetch, "cpb_batch_fetch_cigars")
    refused(lambda: cp.binding._check(lib.cpb_batch_alignment_cigars(b.h, None)), "cpb_batch_alignment_cigars")  # no offsets
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)
    b.ordered_chain(0.85)
    refused(fetch, "cpb_batch_fetch_cigars")  # a decode, no build yet
    want = _check_cigars(b, pairs, "chain")
    # the list stays with its alignment list: reweighting and re-anchoring leave both in place
    b.reweight_pairs(0.5)
    fetch()
    assert np.array_equal(buf[:want[0][-1]], want[1])
    b.anchors_from_alignments(p)
    buf[:] = 0
    fetch()
    assert np.array_equal(buf[:want[0][-1]], want[1])
    # any decode discards it, a refused one too
    b.ordered_chain(0.85)
    refused(fetch, "cpb_batch_fetch_cigars")
    b.alignment_cigars()
    refused(lambda: b.ordered_chain(2.0), "cpb_batch_ordered_chain")
    refused(fetch, "cpb_batch_fetch_cigars")
    refused(build, "cpb_batch_alignment_cigars")  # no alignment list after a refused decode
    # and so does a run
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS_INDELS)
    b.mea(0.5)
    b.alignment_cigars()
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS_INDELS)
    refused(fetch, "cpb_batch_fetch_cigars")
    refused(build, "cpb_batch_alignment_cigars")
    assert lib.cpb_batch_alignment_cigars(b.h, C.c_void_p(off.ctypes.data)) == 2
    b.close()
