"""getMaximalExpectedAccuracyPairwiseAlignment of libcpecan.so (host/realign.c) with its walk-back skipping aligned ranges of the list that
hold no predecessor, against the reference's own function (oracle/_ref, where it is built) and against a plain quadratic restatement of
the reference kept here: the same triples in the same order and the same bits of alignmentScore.  The lists are fuzzed in the reference's
order -- regions ascending, inside a region the traceback blocks last to first, inside a block x + y ascending and x descending -- with
many blocks and several regions, and also shuffled, since the skip is exact in any order.  No GPU involved."""
import ctypes as C

import numpy as np
import pytest

import helpers
from test_realign_host import Host, Ref


class SlabHost(Host):
    """Host, with input lists cut from one slab (cpecan_tripleList_construct) rather than one ctypes call per tuple"""

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


@pytest.fixture(scope="module")
def ref():
    r = helpers.ref_oracle()
    return Ref(r) if r is not None else None


def quadratic_mea(pairs, gapX, gapY, lX, lY, gamma):
    """impl/pairwiseAligner.c:1603-1724 as written: every j < i from i - 1 down, no skipping.  Float and double arithmetic as the C
    evaluates it: the gap terms are int64 * float in float, the first score is float, the candidate a double truncated to int64."""
    g = np.float32(gamma)
    cumX, cumY = np.zeros(max(lX, 1), dtype=np.int64), np.zeros(max(lY, 1), dtype=np.int64)
    for w, x, _ in gapX:
        cumX[x] += w
    for w, _, y in gapY:
        cumY[y] += w
    cumX, cumY = [int(v) for v in np.cumsum(cumX)], [int(v) for v in np.cumsum(cumY)]

    def gap(cum, start, length):
        return 0 if length == 0 else cum[start + length - 1] - (cum[start - 1] if start > 0 else 0)

    def term(v):
        return np.float32(v) * g

    P = [(int(w), int(x), int(y)) for w, x, y in pairs]
    n = len(P)
    scores, back, high = [0.0] * (n + 1), [-1] * (n + 1), [False] * (n + 1)
    best = 0.0
    for i in range(n + 1):
        w, x, y = P[i] if i < n else (0, lX, lY)
        score = float(np.float32(w) + term(gap(cumX, 0, x) + gap(cumY, 0, y)))
        frm = -1
        for j in range(i - 1, -1, -1):
            _, x2, y2 = P[j]
            if x2 < x and y2 < y:
                s = int(float(w) + scores[j] + float(term(gap(cumX, x2 + 1, x - x2 - 1) + gap(cumY, y2 + 1, y - y2 - 1))))
                if s > score:
                    score, frm = float(s), j
                if high[j]:
                    break
        back[i], scores[i] = frm, score
        s = score + float(term((gap(cumX, x + 1, lX - x - 1) if x < lX else 0) + (gap(cumY, y + 1, lY - y - 1) if y < lY else 0)))
        if s >= best:
            best, high[i] = s, True
    out, i = [], back[n]
    while i >= 0:
        out.append(P[i])
        i = back[i]
    return np.array(out[::-1], dtype=np.int64).reshape(-1, 3), best


def reference_order_case(rng, length, regions, blocks, weights="random", per_x=3, band=4):
    """(pairs, gapX, gapY, lX, lY): a posterior cloud near the diagonal of regions that follow each other in x and y, each cut into
    traceback blocks by diagonal, listed as libcpecan.so hands list 0 over"""
    lX, lY = length, length + int(rng.integers(-3, 4))
    cuts = np.sort(rng.choice(np.arange(1, length), regions - 1, replace=False)) if regions > 1 else np.array([], dtype=np.int64)
    bounds = [0] + [int(c) for c in cuts] + [length]
    pairs = []
    for r in range(regions):
        x0, x1 = bounds[r], bounds[r + 1]
        cloud = set()
        for x in range(x0, x1):
            for _ in range(int(rng.integers(0, per_x + 1))):
                y = x + int(rng.integers(-band, band + 1))
                if min(x0, lY) <= y < min(x1, lY):
                    cloud.add((x, y))
        if not cloud:
            continue
        diag = sorted({x + y for x, y in cloud})
        ends = sorted(set(int(v) for v in rng.choice(diag, min(blocks - 1, len(diag)), replace=False))) + [diag[-1]]
        owner = lambda d: next(k for k, e in enumerate(ends) if d <= e)  # noqa: E731
        for k in reversed(range(len(ends))):  # the blocks of a region last to first
            pairs += sorted((p for p in cloud if owner(p[0] + p[1]) == k), key=lambda p: (p[0] + p[1], -p[0]))
    n = len(pairs)
    if weights == "random":
        w = rng.integers(1, 10000001, n)
    elif weights == "ties":  # few distinct weights: many equal candidates
        w = rng.choice([2500000, 5000000, 10000000], n)
    else:  # "negative": reweighted lists can go below 0, and then no isHigh is set before the closing pair
        w = -rng.integers(1, 3000000, n)
    tri = np.array([(int(a), x, y) for a, (x, y) in zip(w, pairs)], dtype=np.int64).reshape(-1, 3)
    gapX = np.array([(int(rng.integers(0, 3000000)), x, int(rng.integers(-1, lY))) for x in range(lX)], dtype=np.int64).reshape(-1, 3)
    gapY = np.array([(int(rng.integers(0, 3000000)), int(rng.integers(-1, lX)), y) for y in range(lY)], dtype=np.int64).reshape(-1, 3)
    return tri, gapX, gapY, lX, lY


def check(host, ref, case, gamma, what, quadratic=True):
    tri, gapX, gapY, lX, lY = case
    got, score = host.mea(tri, gapX, gapY, lX, lY, gamma)
    if quadratic:
        want, want_score = quadratic_mea(tri, gapX, gapY, lX, lY, gamma)
        assert np.array_equal(got, want), "%s: %d triples, restatement %d" % (what, len(got), len(want))
        assert np.float64(score).view(np.int64) == np.float64(want_score).view(np.int64), "%s: %r against %r" % (what, score, want_score)
    if ref is not None:
        want, want_score = ref.mea(tri, gapX, gapY, lX, lY, gamma)
        assert np.array_equal(got, want), what + " (reference build)"
        assert np.float64(score).view(np.int64) == np.float64(want_score).view(np.int64), what + " (reference build)"
    return got


@pytest.mark.parametrize("weights", ["random", "ties", "negative"])
def test_many_blocks_and_regions(host, ref, weights):
    rng = np.random.default_rng({"random": 1, "ties": 2, "negative": 3}[weights])
    for k in range(8):
        length = int(rng.integers(120, 420))
        case = reference_order_case(rng, length, regions=int(rng.integers(1, 5)), blocks=int(rng.integers(2, 12)), weights=weights)
        for gamma in (0.0, 0.5):
            check(host, ref, case, gamma, "%s case %d, gapGamma %g, %d triples" % (weights, k, gamma, len(case[0])))


def test_long_lists_cross_block_summaries(host, ref):
    """lists of several thousand triples, so that whole 1024-triple ranges of later blocks are skipped"""
    rng = np.random.default_rng(9)
    for k, weights in enumerate(("random", "ties", "random")):
        case = reference_order_case(rng, 2000, regions=2 + k, blocks=6, weights=weights)
        assert len(case[0]) > 2048
        check(host, ref, case, 0.5, "long case %d" % k)


def test_no_early_exit(host, ref):
    """negative weights and no gap lists: no pair before the closing one is isHigh, so every walk-back runs to the list's start"""
    rng = np.random.default_rng(4)
    tri, _, _, lX, lY = reference_order_case(rng, 900, regions=3, blocks=5, weights="negative")
    none = np.zeros((0, 3), dtype=np.int64)
    assert len(tri) > 1024
    check(host, ref, (tri, none, none, lX, lY), 0.5, "negative weights, no gaps")
    tri[::7, 0] = 9000000  # some pairs worth taking, none of them isHigh unless it beats every pair before it
    check(host, ref, (tri, none, none, lX, lY), 0.5, "mostly negative weights, no gaps")


@pytest.mark.parametrize("n", [0, 1, 31, 32, 33, 1023, 1024, 1025, 2048])
def test_chunk_boundaries(host, ref, n):
    """lists shorter than one chunk, exactly one chunk or one 1024 range, and one past: taken from a long reference-ordered list"""
    rng = np.random.default_rng(100 + n)
    tri, gapX, gapY, lX, lY = reference_order_case(rng, 1800, regions=2, blocks=7)
    assert len(tri) >= n
    for weights in ("as is", "negative"):
        t = tri[len(tri) - n:].copy() if n else tri[:0].copy()
        if weights == "negative":
            t[:, 0] = -t[:, 0] // 4
        check(host, ref, (t, gapX, gapY, lX, lY), 0.5, "%d triples, %s" % (n, weights))


def test_equal_diagonal_runs_and_ties(host, ref):
    """every pair of a few diagonals, all of one weight, gapGamma 0: candidates tie everywhere and x + y repeats in long runs"""
    lX = lY = 60
    pairs = sorted(((x, y) for x in range(lX) for y in range(lY) if abs(x - y) <= 2), key=lambda p: (p[0] + p[1], -p[0]))
    tri = np.array([(5000000, x, y) for x, y in pairs], dtype=np.int64)
    none = np.zeros((0, 3), dtype=np.int64)
    for gamma in (0.0, 0.9):
        check(host, ref, (tri, none, none, lX, lY), gamma, "ties, gapGamma %g" % gamma)
    half = len(pairs) // 2  # two blocks, the later one first
    blocks = np.concatenate([tri[half:], tri[:half]])
    check(host, ref, (blocks, none, none, lX, lY), 0.0, "ties in two blocks")


def test_empty_inputs(host, ref):
    none = np.zeros((0, 3), dtype=np.int64)
    for lX, lY in ((0, 0), (5, 0), (0, 7), (40, 40)):
        got = check(host, ref, (none, none, none, lX, lY), 0.5, "empty list %d x %d" % (lX, lY))
        assert len(got) == 0


def test_any_order(host, ref):
    """the skip is exact in any list order: shuffled lists and lists sorted by x alone"""
    rng = np.random.default_rng(12)
    for k in range(6):
        tri, gapX, gapY, lX, lY = reference_order_case(rng, int(rng.integers(150, 350)), regions=2, blocks=4)
        order = rng.permutation(len(tri)) if k % 2 == 0 else np.lexsort((tri[:, 2], tri[:, 1]))
        check(host, ref, (tri[order], gapX, gapY, lX, lY), 0.5, "reordered case %d" % k)


@pytest.mark.parametrize("at", [0, 31, 32, 993, 1023, 1024, 1056, 2047, 2080])
def test_lone_predecessor_among_later_pairs(host, ref, at):
    """one early pair (10, 10) at list position `at` among 2 100 pairs of later diagonals, then pairs that follow it: the aligned chunk
    and the 1024 range that hold it must be walked, whatever else they hold"""
    rng = np.random.default_rng(at)
    cells = rng.choice(1000 * 1000, 2100, replace=False)
    later = [(int(rng.integers(1, 1001)), 2000 + int(c) // 1000, 2000 + int(c) % 1000) for c in cells]
    tri = later[:at] + [(9000000, 10, 10)] + later[at:] + [(8000000, 11, 12), (7000000, 13, 13)]
    none = np.zeros((0, 3), dtype=np.int64)
    got = check(host, ref, (np.array(tri, dtype=np.int64), none, none, 3000, 3000), 0.5, "lone predecessor at %d" % at)
    assert [10, 10] in got[:, 1:].tolist()
