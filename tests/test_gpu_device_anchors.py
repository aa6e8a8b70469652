"""Anchors found on the device (cpb_batch_create_anchored, anchor_kernels.cuh) against libcpecan.so's host anchorer
(getBlastPairsForPairwiseAlignmentParameters, host/anchors.c): the same triples in the same order for every pair, and batches made from
them that run exactly as batches made from the host's anchors.  Every comparison is exact."""
import ctypes as C

import numpy as np
import pytest

import cpecan_b200 as cp
import helpers
from cpecan_b200 import synth
from host_anchors import HostAnchorer

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def host():
    return HostAnchorer()


def _rs(rng, n):
    return synth.random_sequence(rng, n, acgt_only=True).encode()


def _mutate(rng, s, rate=0.05):
    a = bytearray(s)
    for i in np.nonzero(rng.random(len(a)) < rate)[0]:
        a[i] = b"ACGT"[(b"ACGT".index(a[i]) + int(rng.integers(1, 4))) % 4]
    return bytes(a)


def _evolved(n, length, seed):
    packed = synth.evolved_pairs(n, length, seed=seed, trim=0, expansion=0)
    return [synth.unpack(packed, i)[:2] for i in range(n)]


def mixed_pairs():
    """(name, sX, sY) covering the anchorer's cases"""
    rng = np.random.default_rng(2024)
    out = []
    for length, n in ((400, 2), (1000, 3), (2000, 2), (12000, 2), (100000, 1)):
        out += [("evolved%d_%d" % (length, i), x, y) for i, (x, y) in enumerate(_evolved(n, length, 17 + length))]
    (x, y), = _evolved(1, 66000, 5)
    out += [("k11", x[:65536], y[:65536]), ("k12", x[:65537], y[:65530])]  # 64 * 65536 = 4^11: the word grows by one base at 65537
    (x, y), = _evolved(1, 20000, 77)
    out.append(("masked", x[:8000] + x[8000:12000].lower() + x[12000:], y))
    out.append(("masked_both", x.lower(), y[:5000] + y[5000:15000].lower() + y[15000:]))
    s = _rs(rng, 2000)
    out.append(("n_run", s[:900] + b"N" * 200 + s[1100:], s))
    out.append(("n_mixed", s[:500] + b"n" * 50 + s[550:1500] + b"xyzN" * 25 + s[1600:], s.lower()))
    out.append(("identical", s, s))
    t = _rs(rng, 12000)
    out.append(("identical12k", t, t))
    out.append(("unrelated", _rs(rng, 3000), _rs(rng, 3000)))
    unit = _rs(rng, 37)
    tandem = unit * 300
    out.append(("tandem", tandem, _mutate(rng, tandem, 0.03)))
    out.append(("tandem_flanked", _rs(rng, 2000) + tandem + _rs(rng, 2000), _rs(rng, 1500) + _mutate(rng, tandem, 0.02) + _rs(rng, 2500)))
    out.append(("short_x", b"ACGTACGTAC", _rs(rng, 30000)))  # a problem shorter than a word
    out.append(("short_y", _rs(rng, 30000), b"ACGTAC"))
    out.append(("empty_x", b"", _rs(rng, 3000)))
    out.append(("empty_y", _rs(rng, 3000), b""))
    out.append(("empty_both", b"", b""))
    # level 2: D's words occur twice in Y, so the whole matrix cannot seed there; the gap around D holds one copy and can
    a, d, c, b = _rs(rng, 6000), _rs(rng, 1500), _rs(rng, 400), _rs(rng, 6000)
    out.append(("level2_repeat", a + d + b, _mutate(rng, a + d + c + b, 0.04) + _mutate(rng, d, 0.04)))
    out.append(("level2_insertion", a + _rs(rng, 3000) + b, _mutate(rng, a + b, 0.04)))
    return out


PAIRS = mixed_pairs()


def param_sets():
    p = cp.pairwiseAlignmentBandingParameters_construct()
    cli = cp.pairwiseAlignmentBandingParameters_construct()
    cli.constraintDiagonalTrim, cli.diagonalExpansion = 0, 4
    small = cp.pairwiseAlignmentBandingParameters_construct()
    small.anchorMatrixBiggerThanThis = 10000
    unmasked = cp.pairwiseAlignmentBandingParameters_construct()
    unmasked.repeatMaskMatrixBiggerThanThis = 10 ** 9
    return {"defaults": p, "cli": cli, "small_matrices": small, "repeat_mask_1e9": unmasked}


def _host_lists(host, pairs, p):
    hp = host.params(p)
    return [host.anchors(x, y, hp) for _, x, y in pairs]


def _check_same(batch, want, pairs):
    off, tri = batch.fetch_anchors()
    assert off[0] == 0 and len(off) == len(pairs) + 1
    for i, (name, _, _) in enumerate(pairs):
        got = tri[off[i]:off[i + 1]]
        assert got.shape == want[i].shape and np.array_equal(got, want[i]), "%s: %d device anchors, %d host anchors" % (
            name, len(got), len(want[i]))


@pytest.mark.parametrize("which", ["defaults", "cli", "small_matrices", "repeat_mask_1e9"])
def test_anchors_equal_the_hosts(ctx, host, which):
    p = param_sets()[which]
    want = _host_lists(host, PAIRS, p)
    b = cp.Batch.anchored(ctx, [x for _, x, _ in PAIRS], [y for _, _, y in PAIRS], p)
    _check_same(b, want, PAIRS)
    b.close()
    names = {n: i for i, (n, _, _) in enumerate(PAIRS)}
    if which == "defaults":  # the cases do what they are there for
        assert len(want[names["evolved400_0"]]) == 0 and len(want[names["evolved100000_0"]]) > 10000
        assert len(want[names["level2_repeat"]]) > 0 and any(1 for x, _, _ in want[names["level2_repeat"]] if 6100 <= x < 7400)
    if which == "repeat_mask_1e9":
        assert any(1 for x, _, _ in want[names["masked"]] if 8100 <= x < 11900)


def test_anchors_equal_the_hosts_in_small_chunks(host):
    """a scratch budget that takes a few problems at a time (the 100 kb pair alone needs about 9 MB)"""
    p = param_sets()["defaults"]
    want = _host_lists(host, PAIRS, p)
    c = cp.Context(0)
    c.set_scratch_budget(12 << 20)
    b = cp.Batch.anchored(c, [x for _, x, _ in PAIRS], [y for _, _, y in PAIRS], p)
    _check_same(b, want, PAIRS)
    b.close()
    c.set_scratch_budget(1 << 20)
    with pytest.raises(cp.CpbError, match="scratch"):
        big = [q for q in PAIRS if q[0] == "evolved100000_0"][0]
        cp.Batch.anchored(c, [big[1]], [big[2]], p)
    c.close()


RUN_PAIRS = [q for q in PAIRS if q[0] in ("evolved1000_0", "evolved1000_1", "evolved2000_0", "evolved12000_0", "evolved12000_1", "masked",
                                          "level2_repeat", "n_run", "identical", "unrelated", "empty_x", "tandem_flanked", "evolved400_0")]


@pytest.mark.parametrize("states", [5, 3])
def test_runs_equal_the_host_anchored_runs(ctx, host, states):
    p = param_sets()["defaults"]
    want = _host_lists(host, RUN_PAIRS, p)
    sx, sy = [x for _, x, _ in RUN_PAIRS], [y for _, _, y in RUN_PAIRS]
    rl = [i % 2 for i in range(len(sx))]
    rr = [(i // 2) % 2 for i in range(len(sx))]
    dev = cp.Batch.anchored(ctx, sx, sy, p, rl, rr)
    ref = cp.Batch(ctx, sx, sy, [w if len(w) else [] for w in want], rl, rr)
    _check_same(dev, want, RUN_PAIRS)
    spec = helpers.ModelSpec(cp.fiveState if states == 5 else cp.threeState)
    for mode in (cp.MODE_ALIGNED_PAIRS, cp.MODE_ALIGNED_PAIRS_INDELS, cp.MODE_EXPECTATIONS, cp.MODE_FORWARD, cp.MODE_ALIGNED_PAIRS):
        for batch in (dev, ref):
            batch.run(spec.cpb(), p, mode)
        if mode in (cp.MODE_ALIGNED_PAIRS, cp.MODE_ALIGNED_PAIRS_INDELS):
            for which in range(3 if mode == cp.MODE_ALIGNED_PAIRS_INDELS else 1):
                for order in (False, True):
                    o1, t1 = dev.fetch_pairs(which, reference_order=order)
                    o2, t2 = ref.fetch_pairs(which, reference_order=order)
                    assert np.array_equal(o1, o2) and np.array_equal(t1, t2), (mode, which, order)
            if mode == cp.MODE_ALIGNED_PAIRS:
                assert np.array_equal(dev.alignment_scores(), ref.alignment_scores())
        elif mode == cp.MODE_EXPECTATIONS:
            pp1, tot1 = dev.fetch_expectations()
            pp2, tot2 = ref.fetch_expectations()
            assert np.array_equal(pp1, pp2) and np.array_equal(tot1, tot2)
        else:
            assert np.array_equal(dev.fetch_forward(), ref.fetch_forward())
    # reweighting, and a second run reusing the plan
    for batch in (dev, ref):
        batch.reweight_pairs(p.gapGamma)
    assert np.array_equal(dev.fetch_pairs(0)[1], ref.fetch_pairs(0)[1])
    assert dev.stats().planReused == ref.stats().planReused
    dev.close()
    ref.close()


def test_python_raw_sequence_forms(ctx, host):
    p = param_sets()["defaults"]
    sM = cp.stateMachine5_construct()
    for name, x, y in PAIRS:
        if name not in ("evolved2000_0", "masked", "level2_repeat"):
            continue
        a = host.anchors(x, y, host.params(p))
        assert cp.getAlignedPairs(sM, x, y, p, ctx=ctx) == cp.getAlignedPairsUsingAnchors(sM, x, y, a, p, ctx=ctx)
        assert cp.getAlignedPairsWithIndels(sM, x, y, p, True, False, ctx=ctx) == cp.getAlignedPairsWithIndelsUsingAnchors(sM, x, y, a, p, True, False,
                                                                                                                          ctx=ctx)
        e1 = cp.getExpectations(sM, np.zeros(cp.hmm_len(5)), x, y, p, ctx=ctx)
        e2 = cp.getExpectationsUsingAnchors(sM, np.zeros(cp.hmm_len(5)), x, y, a, p, ctx=ctx)
        assert np.array_equal(e1, e2)


def test_fetch_anchors_returns_the_callers_own(ctx):
    packed = synth.evolved_pairs(4, 1000, seed=8)
    b = cp.Batch(ctx, None, None, packed=packed)
    off, tri = b.fetch_anchors()
    assert np.array_equal(off, packed["aOff"]) and np.array_equal(tri.reshape(-1), packed["anchors"][:3 * off[-1]])
    b.close()
    b = cp.Batch(ctx, [b"ACGT"], [b"ACGT"])
    off, tri = b.fetch_anchors()
    assert list(off) == [0, 0] and tri.shape == (0, 3)
    b.close()


def test_edge_cases(ctx):
    p = cp.pairwiseAlignmentBandingParameters_construct()
    b = cp.Batch.anchored(ctx, [], [], p)
    off, tri = b.fetch_anchors()
    assert list(off) == [0] and tri.shape == (0, 3)
    b.close()
    bad = {"constraintDiagonalTrim": -1, "diagonalExpansion": -2, "diagonalExpansion ": 1 << 31}
    for field, value in bad.items():
        q = cp.pairwiseAlignmentBandingParameters_construct()
        setattr(q, field.strip(), value)
        h = C.c_void_p()
        xo = np.array([0, 4], dtype=np.int64)
        s = np.frombuffer(b"ACGT", dtype=np.uint8)
        rc = cp.lib.cpb_batch_create_anchored(ctx.h, 1, C.c_void_p(s.ctypes.data), C.c_void_p(xo.ctypes.data), C.c_void_p(s.ctypes.data),
                                              C.c_void_p(xo.ctypes.data), None, None, C.byref(q), C.byref(h))
        assert rc == 2 and not h.value, field  # CPB_ERR_ARGUMENT
