"""Anchors without a subprocess (SURVEY.md section 8f, N3): host/anchors.c of libcpecan.so.

filterToRemoveOverlap and the two-level scheme are the reference's own logic; the filter is compared with the reference build
(oracle/_ref) on fuzzed lists where that build exists, and with its recorded outputs (tests/golden/anchor_lists.json);
getBlastPairs replaces the LASTZ subprocess by an in-process seed-and-chain aligner, whose anchors are checked for what anchors must be: strictly increasing after the filter, inside the matrix, and ON the true alignment of
synthetic evolved pairs.  (What the DP makes of them is checked on the GPU in tests/test_gpu_anchors.py.)
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

import helpers
from cpecan_b200 import synth

LIB = os.environ.get("CPECAN_HOST_LIB") or os.path.join(helpers.ROOT, "cpecan_b200", "lib", "libcpecan.so")
GOLDEN = os.path.join(helpers.ROOT, "tests", "golden", "anchor_lists.json")


class Lists:
    """stList / stIntTuple of one shared library (libcpecan.so's own containers, or the reference build's shim)"""

    def __init__(self, path):
        L = C.CDLL(path)
        for f in ("stList_construct3", "stIntTuple_construct3", "stList_get", "filterToRemoveOverlap", "getBlastPairs",
                  "getBlastPairsForPairwiseAlignmentParameters", "pairwiseAlignmentBandingParameters_construct"):
            if hasattr(L, f):
                getattr(L, f).restype = C.c_void_p
        for f in ("stList_length", "stIntTuple_get"):
            getattr(L, f).restype = C.c_int64
        L.stList_construct3.argtypes = [C.c_int64, C.c_void_p]
        L.stIntTuple_construct3.argtypes = [C.c_int64, C.c_int64, C.c_int64]
        L.stList_append.argtypes = [C.c_void_p, C.c_void_p]
        L.stList_get.argtypes = [C.c_void_p, C.c_int64]
        L.stList_length.argtypes = [C.c_void_p]
        L.stIntTuple_get.argtypes = [C.c_void_p, C.c_int64]
        L.stList_destruct.argtypes = [C.c_void_p]
        L.filterToRemoveOverlap.argtypes = [C.c_void_p]
        self.L = L

    def make(self, triples):
        l = self.L.stList_construct3(0, C.cast(self.L.stIntTuple_destruct, C.c_void_p))
        for a, b, c in triples:
            self.L.stList_append(l, self.L.stIntTuple_construct3(int(a), int(b), int(c)))
        return l

    def read(self, l, free=True):
        n = self.L.stList_length(l)
        out = [(self.L.stIntTuple_get(self.L.stList_get(l, i), 0), self.L.stIntTuple_get(self.L.stList_get(l, i), 1),
                self.L.stIntTuple_get(self.L.stList_get(l, i), 2)) for i in range(n)]
        if free:
            self.L.stList_destruct(l)
        return out


@pytest.fixture(scope="module")
def ours():
    import subprocess

    if not os.path.exists(LIB):
        subprocess.check_call(["make", "-s", "-f", os.path.join(helpers.ROOT, "cpecan_b200", "csrc", "Makefile")])
    return Lists(LIB)


def overlap_cases():
    """300 sorted, overlapping anchor lists (seeded), every fifth with an exact duplicate"""
    rng = np.random.default_rng(5)
    for rep in range(300):
        n = int(rng.integers(0, 60))
        span = int(rng.integers(1, 40))
        t = sorted({(int(rng.integers(0, span)), int(rng.integers(0, span)), int(rng.integers(0, 3))) for _ in range(n)})
        if rep % 5 == 0 and t:
            t = sorted(t + [t[int(rng.integers(0, len(t)))]])  # an exact duplicate
        yield t


def filtered(lists, t):
    a = lists.make(t)
    out = lists.read(lists.L.filterToRemoveOverlap(a))
    lists.L.stList_destruct(a)
    return out


def test_filter_to_remove_overlap_matches_the_reference(ours):
    if helpers.ref_oracle() is None:
        pytest.skip("needs the reference build (oracle/_ref)")
    ref = Lists(helpers.REF_SO)
    for t in overlap_cases():
        got = filtered(ours, t)
        assert got == filtered(ref, t), t
        assert all(p[0] < q[0] and p[1] < q[1] for p, q in zip(got, got[1:]))


def test_filter_to_remove_overlap_matches_the_recorded_lists(ours):
    """the same lists against tests/golden/anchor_lists.json (tools/make_anchor_golden.py), so that the filter is checked where
    the reference build is not"""
    with open(GOLDEN) as f:
        want = json.load(f)["filterToRemoveOverlap"]
    cases = list(overlap_cases())
    assert len(want) == len(cases)
    for t, w in zip(cases, want):
        got = filtered(ours, t)
        assert [list(p) for p in got] == w, t
        assert all(p[0] < q[0] and p[1] < q[1] for p, q in zip(got, got[1:]))


def _true_columns(packed, i):
    """x -> y of the identical aligned columns of pair i (the generator's anchors with trim 0)"""
    _, _, a = synth.unpack(packed, i)
    return {int(x): int(y) for x, y, _ in a}


@pytest.mark.parametrize("length, mask", [(1000, False), (10000, False), (10000, True), (60000, True)])
def test_blast_pairs_lie_on_the_true_alignment(ours, length, mask):
    ours.L.getBlastPairs.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_bool]
    n = 3
    packed = synth.evolved_pairs(n, length, seed=900 + length, trim=0, expansion=0)
    for i in range(n):
        sx, sy, _ = synth.unpack(packed, i)
        truth = _true_columns(packed, i)
        for trim in (0, 14):
            pairs = ours.read(ours.L.getBlastPairs(sx, sy, len(sx), len(sy), trim, 20, mask))
            assert all(0 <= x < len(sx) and 0 <= y < len(sy) and e == 20 for x, y, e in pairs)
            assert all(p[0] < q[0] and p[1] < q[1] for p, q in zip(pairs, pairs[1:])), "one chain: strictly increasing without the filter"
            assert all(p[0] + p[1] <= q[0] + q[1] for p, q in zip(pairs, pairs[1:]))
            known = [(x, y) for x, y, _ in pairs if x in truth]
            wrong = sum(1 for x, y in known if truth[x] != y)
            assert len(known) > len(sx) * (0.08 if trim else 0.3), "anchors cover a good part of the pair (%d of %d)" % (len(known), len(sx))
            # next to an indel the placement of the gap is ambiguous (a base of the run may match on either side), and a deletion
            # followed closely by an insertion of the same length leaves a stretch that a gapless run bridges on the straight diagonal:
            # such columns are off the generator's alignment by a position or two, far inside any band
            assert wrong <= 0.01 * len(known), "%d of %d anchors off the true alignment" % (wrong, len(known))
            off = [abs(truth[x] - y) for x, y in known if truth[x] != y]
            assert not off or max(off) <= 8  # two indels of up to four bases each


def test_blast_pairs_edge_cases(ours):
    ours.L.getBlastPairs.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_bool]
    assert ours.read(ours.L.getBlastPairs(b"", b"ACGT", 0, 4, 0, 4, False)) == []
    assert ours.read(ours.L.getBlastPairs(b"ACGTACGT", b"ACG", 8, 3, 0, 4, False)) == []  # shorter than a word
    rng = np.random.default_rng(3)
    def rs(n):
        return synth.random_sequence(rng, n, acgt_only=True).encode()

    a, b = rs(3000), rs(3000)
    assert len(ours.read(ours.L.getBlastPairs(a, b, 3000, 3000, 0, 4, False))) == 0  # unrelated sequences: nothing to anchor on
    s = rs(2000)
    same = ours.read(ours.L.getBlastPairs(s, s, 2000, 2000, 0, 6, False))
    assert same == [(i, i, 6) for i in range(2000)]  # identical sequences: the whole diagonal
    low = ours.read(ours.L.getBlastPairs(s.lower(), s.lower(), 2000, 2000, 0, 6, True))
    assert low == []  # soft-masked everywhere: no seeds (the reference leaves lower case to LASTZ's masking)
    assert ours.read(ours.L.getBlastPairs(s.lower(), s, 2000, 2000, 0, 6, False)) == same  # without masking case does not matter
    n_runs = ours.read(ours.L.getBlastPairs(s[:900] + b"N" * 200 + s[1100:], s, 2000, 2000, 0, 6, False))
    assert all(x == y for x, y, _ in n_runs) and not any(900 <= x < 1100 for x, _, _ in n_runs)


def test_two_level_scheme(ours):
    """getBlastPairsForPairwiseAlignmentParameters: nothing below anchorMatrixBiggerThanThis; above it the combined list is
    strictly increasing, and a gap that is itself a big matrix gets anchors of its own"""
    L = ours.L

    class Params(C.Structure):
        _fields_ = [("threshold", C.c_double), ("minDiagsBetweenTraceBack", C.c_int64), ("traceBackDiagonals", C.c_int64),
                    ("diagonalExpansion", C.c_int64), ("constraintDiagonalTrim", C.c_int64), ("anchorMatrixBiggerThanThis", C.c_int64),
                    ("repeatMaskMatrixBiggerThanThis", C.c_int64), ("splitMatrixBiggerThanThis", C.c_int64),
                    ("alignAmbiguityCharacters", C.c_bool), ("gapGamma", C.c_float), ("dynamicAnchorExpansion", C.c_bool)]

    L.getBlastPairsForPairwiseAlignmentParameters.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int64, C.c_void_p]
    p = C.cast(L.pairwiseAlignmentBandingParameters_construct(), C.POINTER(Params))
    rng = np.random.default_rng(9)
    s = synth.random_sequence(rng, 400, acgt_only=True).encode()
    assert ours.read(L.getBlastPairsForPairwiseAlignmentParameters(s, s, 400, 400, p)) == []  # 160 000 <= 250 000: unanchored
    packed = synth.evolved_pairs(1, 20000, seed=77, trim=0, expansion=0)
    sx, sy, _ = synth.unpack(packed, 0)
    # lower-case a stretch of X: the top level (soft-masked) cannot seed there, the gap is anchored again without the mask
    sx = sx[:8000] + sx[8000:12000].lower() + sx[12000:]
    truth = _true_columns(packed, 0)
    pairs = ours.read(L.getBlastPairsForPairwiseAlignmentParameters(sx, sy, len(sx), len(sy), p))
    assert not [1 for x, _, _ in pairs if 8100 <= x < 11900]  # with the defaults a gap this big is anchored with the mask on again (:1148)
    p.contents.repeatMaskMatrixBiggerThanThis = 10 ** 9
    pairs = ours.read(L.getBlastPairsForPairwiseAlignmentParameters(sx, sy, len(sx), len(sy), p))
    assert all(a[0] < b[0] and a[1] < b[1] for a, b in zip(pairs, pairs[1:]))
    inside = [(x, y) for x, y, _ in pairs if 8100 <= x < 11900]
    assert len(inside) > 600, "the masked stretch was anchored by the second level (%d anchors)" % len(inside)
    known = [(x, y) for x, y, _ in pairs if x in truth]
    assert sum(1 for x, y in known if truth[x] != y) <= 0.01 * len(known)
