"""Host-side list work of libcpecan.so after the device pass (cpecan_b200/csrc/host/realign.c, bioio.c): anchors from cigars,
gap reweighting, scores, the maximal-expected-accuracy alignment, left shift and the heaviest ordered chain, plus cigar / FASTA I/O.

Checked (i) live against the reference's own functions in oracle/_ref (impl/pairwiseAligner.c:979-1003, :1519-1792 compiled
unmodified) where that build exists, (ii) against tests/golden/realign_cases.json, generated from the same reference build by
tools/make_realign_golden.py, and for the anchors from cigars against this library's recorded outputs (tests/golden/anchor_lists.json,
tools/make_anchor_golden.py), and (iii) the chain -- which the reference computes inside its multiple aligner with randomised
weights -- against a quadratic dynamic programme.  No GPU involved.
"""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

import helpers

ROOT = helpers.ROOT
HOST_SO = os.path.join(ROOT, "cpecan_b200", "lib", "libcpecan.so")
GOLDEN = os.path.join(ROOT, "tests", "golden", "realign_cases.json")


class PairwiseAlignmentParameters(C.Structure):
    """include/cpecan/pairwiseAligner.h (inc/pairwiseAligner.h:28-41 of the reference)"""
    _fields_ = [("threshold", C.c_double), ("minDiagsBetweenTraceBack", C.c_int64), ("traceBackDiagonals", C.c_int64),
                ("diagonalExpansion", C.c_int64), ("constraintDiagonalTrim", C.c_int64), ("anchorMatrixBiggerThanThis", C.c_int64),
                ("repeatMaskMatrixBiggerThanThis", C.c_int64), ("splitMatrixBiggerThanThis", C.c_int64), ("alignAmbiguityCharacters", C.c_bool),
                ("gapGamma", C.c_float), ("dynamicAnchorExpansion", C.c_bool)]


class Host:
    """ctypes view of the sonLib-style list API and the realign functions of libcpecan.so"""

    def __init__(self):
        if not os.path.exists(HOST_SO):
            subprocess.check_call(["make", "-s", "-f", os.path.join(ROOT, "cpecan_b200", "csrc", "Makefile")])
        L = self.L = C.CDLL(HOST_SO)
        vp, i64 = C.c_void_p, C.c_int64
        L.stList_construct3.restype = vp
        L.stList_construct3.argtypes = [i64, vp]
        L.stList_append.argtypes = [vp, vp]
        L.stList_length.restype = i64
        L.stList_length.argtypes = [vp]
        L.stList_get.restype = vp
        L.stList_get.argtypes = [vp, i64]
        L.stList_destruct.argtypes = [vp]
        L.stIntTuple_construct3.restype = vp
        L.stIntTuple_construct3.argtypes = [i64, i64, i64]
        L.stIntTuple_get.restype = i64
        L.stIntTuple_get.argtypes = [vp, i64]
        L.stIntTuple_length.restype = i64
        L.stIntTuple_length.argtypes = [vp]
        L.reweightAlignedPairs2.restype = vp
        L.reweightAlignedPairs2.argtypes = [vp, i64, i64, C.c_double]
        for name in ("scoreByIdentity", "scoreByIdentityIgnoringGaps", "scoreByPosteriorProbability", "scoreByPosteriorProbabilityIgnoringGaps"):
            getattr(L, name).restype = C.c_double
        L.scoreByIdentity.argtypes = [C.c_char_p, C.c_char_p, i64, i64, vp]
        L.scoreByIdentityIgnoringGaps.argtypes = [C.c_char_p, C.c_char_p, vp]
        L.scoreByPosteriorProbability.argtypes = [i64, i64, vp]
        L.scoreByPosteriorProbabilityIgnoringGaps.argtypes = [vp]
        L.getMaximalExpectedAccuracyPairwiseAlignment.restype = vp
        L.getMaximalExpectedAccuracyPairwiseAlignment.argtypes = [vp, vp, vp, i64, i64, C.POINTER(C.c_double), vp]
        L.leftShiftAlignment.restype = vp
        L.leftShiftAlignment.argtypes = [vp, C.c_char_p, C.c_char_p]
        L.filterPairwiseAlignmentToMakePairsOrdered.restype = vp
        L.filterPairwiseAlignmentToMakePairsOrdered.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_float]
        L.pairwiseAlignmentBandingParameters_construct.restype = vp
        L.pairwiseAlignmentBandingParameters_destruct.argtypes = [vp]
        self.tupleDestructor = C.cast(L.stIntTuple_destruct, vp)

    def to_list(self, triples):
        l = self.L.stList_construct3(0, self.tupleDestructor)
        for t in np.asarray(triples, dtype=np.int64).reshape(-1, 3):
            self.L.stList_append(l, self.L.stIntTuple_construct3(int(t[0]), int(t[1]), int(t[2])))
        return l

    def from_list(self, l, destruct=True):
        n = self.L.stList_length(l)
        out = np.zeros((n, 3), dtype=np.int64)
        for i in range(n):
            t = self.L.stList_get(l, i)
            for k in range(3):
                out[i, k] = self.L.stIntTuple_get(t, k)
        if destruct:
            self.L.stList_destruct(l)
        return out

    def reweight(self, pairs, lX, lY, gamma):
        return self.from_list(self.L.reweightAlignedPairs2(self.to_list(pairs), lX, lY, gamma))

    def scores(self, sX, sY, pairs):
        l = self.to_list(pairs)
        bx, by = sX.encode(), sY.encode()
        out = [self.L.scoreByIdentity(bx, by, len(sX), len(sY), l), self.L.scoreByIdentityIgnoringGaps(bx, by, l),
               self.L.scoreByPosteriorProbability(len(sX), len(sY), l), self.L.scoreByPosteriorProbabilityIgnoringGaps(l)]
        self.L.stList_destruct(l)
        return out

    def mea(self, pairs, gapX, gapY, lX, lY, gamma):
        p = self.L.pairwiseAlignmentBandingParameters_construct()
        C.cast(p, C.POINTER(PairwiseAlignmentParameters)).contents.gapGamma = gamma
        a, x, y = self.to_list(pairs), self.to_list(gapX), self.to_list(gapY)
        score = C.c_double()
        out = self.from_list(self.L.getMaximalExpectedAccuracyPairwiseAlignment(a, x, y, lX, lY, C.byref(score), p))
        for l in (a, x, y):
            self.L.stList_destruct(l)
        self.L.pairwiseAlignmentBandingParameters_destruct(p)
        return out, score.value

    def left_shift(self, pairs, sX, sY):
        a = self.to_list(pairs)
        out = self.from_list(self.L.leftShiftAlignment(a, sX.encode(), sY.encode()))
        self.L.stList_destruct(a)
        return out

    def chain(self, pairs, sX, sY, matchGamma):
        return self.from_list(self.L.filterPairwiseAlignmentToMakePairsOrdered(self.to_list(pairs), sX.encode(), sY.encode(), matchGamma))


@pytest.fixture(scope="module")
def host():
    return Host()


def random_case(rng, n=None):
    """sequences plus a cloud of weighted pairs near the diagonal, in the engine's order, and gap lists"""
    lX = int(rng.integers(1, 60)) if n is None else n
    lY = max(1, lX + int(rng.integers(-5, 6)))
    sX = "".join(rng.choice(list("ACGTN"), lX, p=[0.24, 0.24, 0.24, 0.24, 0.04]))
    sY = "".join(rng.choice(list("ACGTacgt"), lY))
    seen = set()
    for x in range(lX):
        for _ in range(int(rng.integers(0, 4))):
            y = x + int(rng.integers(-3, 4))
            if 0 <= y < lY:
                seen.add((x, y))
    pairs = sorted(seen, key=lambda t: (t[0] + t[1], -t[0]))  # diagonals ascending, x descending: one traceback block of the reference
    tri = np.array([(int(rng.integers(1, 10000001)), x, y) for x, y in pairs], dtype=np.int64).reshape(-1, 3)
    gapX = np.array([(int(rng.integers(0, 3000000)), x, int(rng.integers(-1, lY))) for x in range(lX)], dtype=np.int64).reshape(-1, 3)
    gapY = np.array([(int(rng.integers(0, 3000000)), int(rng.integers(-1, lX)), y) for y in range(lY)], dtype=np.int64).reshape(-1, 3)
    return sX, sY, tri, gapX, gapY


class Ref:
    """the reference's own functions through oracle/ref_driver.c"""

    def __init__(self, oracle):
        self.L = oracle.L
        self.L.orc_scores.restype = None
        self.L.orc_reweight.restype = C.c_int64
        self.L.orc_mea.restype = C.c_int64
        self.L.orc_left_shift.restype = C.c_int64
        self.L.orc_cigar_anchors.restype = C.c_int64

    @staticmethod
    def _p(a):
        return a.ctypes.data_as(C.POINTER(C.c_int64))

    def reweight(self, pairs, lX, lY, gamma):
        pairs = np.ascontiguousarray(pairs, dtype=np.int64)
        out = np.zeros_like(pairs)
        n = self.L.orc_reweight(self._p(pairs), C.c_int64(len(pairs)), C.c_int64(lX), C.c_int64(lY), C.c_double(gamma), self._p(out))
        return out[:n]

    def scores(self, sX, sY, pairs):
        pairs = np.ascontiguousarray(pairs, dtype=np.int64)
        out = np.zeros(4)
        self.L.orc_scores(sX.encode(), sY.encode(), self._p(pairs), C.c_int64(len(pairs)), out.ctypes.data_as(C.POINTER(C.c_double)))
        return list(out)

    def mea(self, pairs, gapX, gapY, lX, lY, gamma):
        pairs, gapX, gapY = (np.ascontiguousarray(a, dtype=np.int64) for a in (pairs, gapX, gapY))
        out = np.zeros((len(pairs) + 1, 3), dtype=np.int64)
        score = C.c_double()
        n = self.L.orc_mea(self._p(pairs), C.c_int64(len(pairs)), self._p(gapX), C.c_int64(len(gapX)), self._p(gapY), C.c_int64(len(gapY)),
                           C.c_int64(lX), C.c_int64(lY), C.c_double(gamma), self._p(out), C.byref(score))
        return out[:n], score.value

    def left_shift(self, pairs, sX, sY):
        pairs = np.ascontiguousarray(pairs, dtype=np.int64)
        cap = len(pairs) + len(sX) + len(sY) + 4
        out = np.zeros((cap, 3), dtype=np.int64)
        n = self.L.orc_left_shift(self._p(pairs), C.c_int64(len(pairs)), sX.encode(), sY.encode(), self._p(out), C.c_int64(cap))
        return out[:n]

    def cigar_anchors(self, ops, start1, start2, trim, expansion):
        ops = np.ascontiguousarray(ops, dtype=np.int64)
        cap = int(ops[:, 1].sum()) + 1
        out = np.zeros((cap, 3), dtype=np.int64)
        n = self.L.orc_cigar_anchors(self._p(ops), C.c_int64(len(ops)), C.c_int64(start1), C.c_int64(start2), C.c_int64(trim), C.c_int64(expansion),
                                     self._p(out), C.c_int64(cap))
        return out[:n]


def increasing_chain(pairs):
    return all(a[1] < b[1] and a[2] < b[2] for a, b in zip(pairs[:-1], pairs[1:]))


def all_results(host_or_ref, case, gamma=0.5):
    sX, sY, tri, gapX, gapY = case
    rw = host_or_ref.reweight(tri, len(sX), len(sY), gamma)
    mea, score = host_or_ref.mea(tri, gapX, gapY, len(sX), len(sY), gamma)
    return {"reweighted": rw.tolist(), "scores": [float(v) for v in host_or_ref.scores(sX, sY, tri)], "mea": mea.tolist(), "mea_score": float(score),
            "left_shift": host_or_ref.left_shift(mea, sX, sY).tolist()}


def assert_same(got, want, what):
    assert got["reweighted"] == want["reweighted"], what
    assert got["mea"] == want["mea"], what
    assert got["mea_score"] == want["mea_score"], what  # same float / int64 arithmetic, operation for operation
    assert got["left_shift"] == want["left_shift"], what
    np.testing.assert_allclose(got["scores"], want["scores"], rtol=1e-15, atol=0, err_msg=what)


def test_list_functions_match_the_reference_build_live(host):
    ref = helpers.ref_oracle()
    if ref is None:
        pytest.skip("oracle/_ref not built here (no /root/reference); the golden fixture covers this")
    ref = Ref(ref)
    rng = np.random.default_rng(77)
    for i in range(60):
        case = random_case(rng)
        gamma = [0.0, 0.2, 0.5, 0.9][i % 4]
        assert_same(all_results(host, case, gamma), all_results(ref, case, gamma), "case %d" % i)


def test_list_functions_match_the_golden_fixture(host):
    cases = json.load(open(GOLDEN))["cases"]
    assert len(cases) >= 10
    for i, c in enumerate(cases):
        case = (c["sX"], c["sY"], np.array(c["pairs"], dtype=np.int64).reshape(-1, 3), np.array(c["gapX"], dtype=np.int64).reshape(-1, 3),
                np.array(c["gapY"], dtype=np.int64).reshape(-1, 3))
        assert_same(all_results(host, case, c["gamma"]), c["want"], "golden case %d" % i)


def test_chain_is_the_heaviest_ordered_subset(host):
    """filterPairwiseAlignmentToMakePairsOrdered (impl/multipleAligner.c:945-972): strictly increasing in x and y, only pairs of
    weight >= matchGamma, and no heavier such chain exists (quadratic DP)."""
    rng = np.random.default_rng(5)
    for i in range(40):
        sX, sY, tri, _, _ = random_case(rng)
        gamma = [0.0, 0.3, 0.85][i % 3]
        got = host.chain(tri, sX, sY, gamma)
        assert increasing_chain(got)
        allowed = {(int(t[1]), int(t[2])): int(t[0]) for t in tri if t[0] / 1e7 >= np.float32(gamma) and t[0] > 0}
        for t in got:
            assert allowed[(int(t[1]), int(t[2]))] == int(t[0])
        cand = sorted((x, y, w) for (x, y), w in allowed.items())
        best = [0] * len(cand)
        for a, (x, y, w) in enumerate(cand):
            best[a] = w + max([best[b] for b in range(a) if cand[b][0] < x and cand[b][1] < y], default=0)
        assert int(got[:, 0].sum()) == max(best, default=0), "case %d" % i


def test_chain_of_nothing_and_of_one(host):
    assert host.chain(np.zeros((0, 3)), "ACGT", "ACGT", 0.85).shape == (0, 3)
    assert host.chain(np.array([[9000000, 2, 1]]), "ACGT", "ACGT", 0.85).tolist() == [[9000000, 2, 1]]
    assert host.chain(np.array([[8000000, 2, 1]]), "ACGT", "ACGT", 0.85).shape == (0, 3)


def cigar_cases():
    """30 seeded alignments as (operations, start1, start2, trim, expansion)"""
    rng = np.random.default_rng(11)
    for _ in range(30):
        ops = np.array([(int(rng.integers(0, 3)), int(rng.integers(1, 12))) for _ in range(int(rng.integers(1, 9)))], dtype=np.int64)
        s1, s2, trim, e = int(rng.integers(0, 50)), int(rng.integers(0, 50)), int(rng.integers(0, 4)), 2 * int(rng.integers(0, 6))
        yield ops, s1, s2, trim, e


def host_cigar_anchors(host, ops, s1, s2, trim, e):
    """convertPairwiseForwardStrandAlignmentToAnchorPairs of libcpecan.so on one alignment"""
    L = host.L
    vp, i64 = C.c_void_p, C.c_int64
    L.constructEmptyList.restype = vp
    L.constructEmptyList.argtypes = [i64, vp]
    L.listAppend.argtypes = [vp, vp]
    L.constructAlignmentOperation.restype = vp
    L.constructAlignmentOperation.argtypes = [i64, i64, C.c_double]
    L.constructPairwiseAlignment.restype = vp
    L.constructPairwiseAlignment.argtypes = [C.c_char_p, i64, i64, i64, C.c_char_p, i64, i64, i64, C.c_double, vp]
    L.destructPairwiseAlignment.argtypes = [vp]
    L.convertPairwiseForwardStrandAlignmentToAnchorPairs.restype = vp
    L.convertPairwiseForwardStrandAlignmentToAnchorPairs.argtypes = [vp, i64, i64]
    opList = L.constructEmptyList(0, C.cast(L.destructAlignmentOperation, vp))
    for t, n in ops:
        L.listAppend(opList, L.constructAlignmentOperation(int(t), int(n), 0.0))  # 0 match, 1 indel X, 2 indel Y (cpecan/pairwiseAlignment.h)
    e1 = s1 + int(ops[ops[:, 0] != 2, 1].sum())
    e2 = s2 + int(ops[ops[:, 0] != 1, 1].sum())
    pA = L.constructPairwiseAlignment(b"a", s1, e1, 1, b"b", s2, e2, 1, 0.0, opList)
    got = host.from_list(L.convertPairwiseForwardStrandAlignmentToAnchorPairs(pA, trim, e))
    L.destructPairwiseAlignment(pA)
    return got


def test_cigar_anchors_match_the_reference(host):
    ref = helpers.ref_oracle()
    if ref is None:
        pytest.skip("oracle/_ref not built here")
    ref = Ref(ref)
    for case in cigar_cases():
        assert host_cigar_anchors(host, *case).tolist() == ref.cigar_anchors(*case).tolist()


def test_cigar_anchors_match_the_recorded_lists(host):
    """the same alignments against tests/golden/anchor_lists.json (tools/make_anchor_golden.py), so that the conversion is checked
    where the reference build is not"""
    want = json.load(open(os.path.join(ROOT, "tests", "golden", "anchor_lists.json")))["cigarAnchors"]
    cases = list(cigar_cases())
    assert len(want) == len(cases)
    for case, w in zip(cases, want):
        assert host_cigar_anchors(host, *case).tolist() == w


CIGARS = """cigar: b 0 10 + a 5 16 + 57.500000 M 4 D 1 M 6
# a comment line
cigar: seq2 30 10 - seq1 100 125 + 0.000000 M 10 I 5 M 5 D 10
"""


def test_cigar_and_fasta_round_trip(tmp_path):
    """cigarRead / cigarWrite / fastaReadToFunction of libcpecan.so through a small C driver: query-first field order,
    M / D / I operations, strands, '%f' scores (the format LASTZ --format=cigar writes and cPecanRealign.c:509, :591-599 exchange)."""
    src = tmp_path / "io.c"
    src.write_text(r'''
#include <inttypes.h>
#include <stdio.h>
#include "cpecan/pairwiseAlignment.h"
static void show(const char *h, const char *s, int64_t n) { printf("seq [%s] %" PRIi64 " %s\n", h, n, s); }
int main(int argc, char **argv) {
    FILE *f = fopen(argv[1], "r");
    struct PairwiseAlignment *pA;
    while ((pA = cigarRead(f)) != NULL) {
        checkPairwiseAlignment(pA);
        printf("read %s %" PRIi64 " %" PRIi64 " %" PRIi64 " | %s %" PRIi64 " %" PRIi64 " %" PRIi64 " | %" PRIi64 " ops\n", pA->contig1, pA->start1, pA->end1, pA->strand1,
               pA->contig2, pA->start2, pA->end2, pA->strand2, pA->operationList->length);
        cigarWrite(stdout, pA, 0);
        destructPairwiseAlignment(pA);
    }
    fclose(f);
    f = fopen(argv[2], "r");
    fastaReadToFunction(f, show);
    fclose(f);
    char *rc = stString_reverseComplementString("ACGTNacgtR");
    printf("rc %s\n", rc);
    return 0;
}
''')
    (tmp_path / "in.cig").write_text(CIGARS)
    (tmp_path / "in.fa").write_text(">one first record\nACGT\nAC GT\n\n>two\n>three\tx\nNNNN\nacgt")
    exe = tmp_path / "io"
    lib = os.path.dirname(HOST_SO)
    subprocess.check_call(["gcc", "-std=c99", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe), "-L" + lib, "-lcpecan", "-lcpecan_b200",
                           "-Wl,-rpath," + lib, "-lm"])
    out = subprocess.check_output([str(exe), str(tmp_path / "in.cig"), str(tmp_path / "in.fa")], text=True).splitlines()
    assert out[0] == "read a 5 16 1 | b 0 10 1 | 3 ops"
    assert out[1] == "cigar: b 0 10 + a 5 16 + 57.500000 M 4 D 1 M 6"
    assert out[2] == "read seq1 100 125 1 | seq2 30 10 0 | 4 ops"
    assert out[3] == "cigar: seq2 30 10 - seq1 100 125 + 0.000000 M 10 I 5 M 5 D 10"
    assert out[4:7] == ["seq [one first record] 8 ACGTACGT", "seq [two] 0 ", "seq [three\tx] 8 NNNNacgt"]
    assert out[7] == "rc YacgtNACGT"
    # the same files with DOS line ends read the same
    (tmp_path / "dos.cig").write_bytes(CIGARS.replace("\n", "\r\n").encode())
    (tmp_path / "dos.fa").write_bytes(b">one first record\r\nACGT\r\nAC GT\r\n\r\n>two\r\n>three\tx\r\nNNNN\r\nacgt")
    assert subprocess.check_output([str(exe), str(tmp_path / "dos.cig"), str(tmp_path / "dos.fa")], text=True).splitlines() == out


LIB_DIR = os.path.dirname(HOST_SO)


def test_programs_print_their_options_without_a_gpu():
    for exe, needle in (("cPecanRealign", "--outputExpectations"), ("cPecanEm", "--trainEmissions")):
        out = subprocess.run([os.path.join(LIB_DIR, exe), "--help"], capture_output=True, text=True)
        assert out.returncode == 0 and needle in out.stderr, exe


def test_programs_fail_loudly_without_a_gpu(tmp_path):
    """no CPU implementation of the DP behind the command line either: without a CUDA device the programs abort with the engine's message"""
    import torch

    if torch.cuda.is_available():
        pytest.skip("needs a box without a GPU")
    fa = tmp_path / "s.fa"
    fa.write_text(">a\nACGTACGTAC\n>b\nACGTTCGTAC\n")
    cig = "cigar: b 0 10 + a 0 10 + 0 M 10\n"
    for exe, args in (("cPecanRealign", []), ("cPecanEm", ["--iterations", "1", "--outputModel", str(tmp_path / "m.hmm")])):
        out = subprocess.run([os.path.join(LIB_DIR, exe)] + args + [str(fa)], input=cig, capture_output=True, text=True)
        assert out.returncode != 0, exe
        assert "CUDA" in out.stderr or "no CPU implementation" in out.stderr, out.stderr


def test_malformed_input_is_an_error(tmp_path):
    """sonLib's convention: print a message and exit (st_errAbort), never a silent partial result"""
    fa = tmp_path / "s.fa"
    fa.write_text(">a\nACGTACGTAC\n>b\nACGTTCGTAC\n")
    exe = os.path.join(LIB_DIR, "cPecanRealign")
    for cig, needle in (("cigar: b 0 10 + a 0 10 + 0 M 9\n", "operations cover"),      # lengths do not add up
                        ("cigar: b 0 10 + a 0 10 + 0 Q 10\n", "operation 'Q'"),        # unknown operation
                        ("cigar: b 0 10 + a 0 10\n", "leading fields"),                # truncated line
                        ("cigar: b 0 10 + a 0 40 + 0 M 10 D 30\n", "beyond the end")): # past the end of the sequence
        out = subprocess.run([exe, str(fa)], input=cig, capture_output=True, text=True)
        assert out.returncode != 0 and needle in out.stderr, (cig, out.stderr)
