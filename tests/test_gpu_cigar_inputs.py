"""Cigars in on the device: a batch anchored from input cigars (cpb_batch_create_from_cigars) and an alignment list made of a cigar's columns
weighed against list 0 (cpb_batch_alignments_from_cigars); k_cigar_cols_count, k_cigar_cols_write and k_cigar_weigh of decode_kernels.cuh.

The definitions are the host's: the anchors are libcpecan.so's convertPairwiseForwardStrandAlignmentToAnchorPairs followed by job_prepare's
columns_match filter (host/realignJobs.h); the weighed list is cPecanRealign's score_anchor_pairs, put in x order.  Every comparison is
exact.  Neither entry point needs a work array, so there is no scratch budget for a pair to exceed."""
import ctypes as C

import numpy as np
import pytest

import cpecan_b200 as cp
from test_gpu_alignments import PAIRS, SlabHost, _batch, _model, _per_pair, _same_bits, param_sets
from test_gpu_band_update import _assert_same_outputs, _outputs, _fresh, with_band
from test_gpu_realign_cli import cigar_line, cli_params, make_inputs, ops_from_columns
from test_gpu_realign_device import run, score_text
from test_realign_host import host_cigar_anchors

pytestmark = pytest.mark.gpu

BIG_TRIM = 1 << 20  # more than every operation's length: no columns at all


@pytest.fixture(scope="module")
def host():
    return SlabHost()


@pytest.fixture
def keep():
    """keep(batch) -> batch, closed when the test ends, whether it passes or not (before the session's context goes)"""
    made = []

    def add(b):
        made.append(b)
        return b

    yield add
    for b in made:
        b.close()


def packed(op_lists):
    """[[(type, length), ...] per pair] -> (offsets[n+1] int64, ops[m, 2] int32), the form Batch.alignment_cigars returns"""
    off = np.zeros(len(op_lists) + 1, dtype=np.int64)
    np.cumsum([len(o) for o in op_lists], out=off[1:])
    return off, np.array([o for ops in op_lists for o in ops], dtype=np.int32).reshape(-1, 2)


def unpacked(cigars):
    off, ops = cigars
    return [[(int(t), int(n)) for t, n in ops[off[i]:off[i + 1]]] for i in range(len(off) - 1)]


def host_columns(host, ops, trim):
    """convertPairwiseForwardStrandAlignmentToAnchorPairs of libcpecan.so: the (x, y) of every MATCH column at [trim, L - trim)"""
    return host_cigar_anchors(host, np.array(ops, dtype=np.int64).reshape(-1, 2), 0, 0, trim, 0)[:, :2]


def host_anchors(host, ops, sX, sY, trim, expansion):
    """job_prepare's filtered anchors of a cigar over the whole of sX and sY"""
    cols = host_columns(host, ops, trim)
    ux, uy = np.frombuffer(cp.binding._as_bytes(sX).upper(), dtype=np.uint8), np.frombuffer(cp.binding._as_bytes(sY).upper(), dtype=np.uint8)
    if len(cols) == 0:
        return np.zeros((0, 3), dtype=np.int64)
    cx, cy = ux[cols[:, 0]], uy[cols[:, 1]]
    kept = cols[(cx == cy) & (cx != ord("N"))]
    return np.concatenate([kept, np.full((len(kept), 1), expansion, dtype=np.int64)], axis=1)


def host_weighed(cols, list0):
    """score_anchor_pairs of cPecanRealign with list 0 as a dict: the columns found in list 0 with their weights, in list 0's order, then
    the others with weight 0 in column order"""
    index = {(int(x), int(y)): k for k, (x, y) in enumerate(cols)}
    seen = np.zeros(len(cols), dtype=bool)
    out = []
    for w, x, y in list0:
        k = index.get((int(x), int(y)))
        if k is not None:
            seen[k] = True
            out.append((int(w), int(x), int(y)))
    out += [(0, int(x), int(y)) for k, (x, y) in enumerate(cols) if not seen[k]]
    return np.array(out, dtype=np.int64).reshape(-1, 3)


# ---- cigars and their perturbations: the same walk, other operations ----
def split_runs(ops, rng):
    """MATCH runs split into adjacent MATCH operations, zero-length operations of every type, INDEL_Y before INDEL_X"""
    out = [(cp.OP_MATCH, 0), (cp.OP_INDEL_X, 0), (cp.OP_INDEL_Y, 0)]
    for t, n in ops:
        if t == cp.OP_MATCH and n >= 2 and rng.random() < 0.6:
            k = int(rng.integers(1, n))
            out += [(t, k), (t, n - k)]
        else:
            out.append((t, n))
        if rng.random() < 0.3:
            out.append((int(rng.integers(0, 3)), 0))
    k = 0
    while k + 1 < len(out):
        if out[k][0] == cp.OP_INDEL_X and out[k + 1][0] == cp.OP_INDEL_Y:
            out[k], out[k + 1] = out[k + 1], out[k]
            k += 2
        else:
            k += 1
    return out + [(cp.OP_INDEL_Y, 0)]


def end_indels(ops):
    """the first and the last column of the alignment as an INDEL_X and an INDEL_Y each: leading and trailing indels"""
    out = list(ops)
    first = next((k for k, (t, n) in enumerate(out) if t == cp.OP_MATCH and n > 0), None)
    if first is None:
        return out
    out[first:first + 1] = [(cp.OP_INDEL_X, 1), (cp.OP_INDEL_Y, 1), (cp.OP_MATCH, out[first][1] - 1)]
    last = max(k for k, (t, n) in enumerate(out) if t == cp.OP_MATCH)
    if out[last][1] > 0:
        out[last:last + 1] = [(cp.OP_MATCH, out[last][1] - 1), (cp.OP_INDEL_Y, 1), (cp.OP_INDEL_X, 1)]
    return out


def all_indels(lX, lY, y_first):
    ops = [(cp.OP_INDEL_X, lX), (cp.OP_INDEL_Y, lY)]
    return ops[::-1] if y_first else ops


def variants(seqs, op_lists, seed):
    """every pair with its cigar, perturbed in each way -> (sX list, sY list, op lists)"""
    rng = np.random.default_rng(seed)
    sx, sy, cig = [], [], []
    for k, ((a, b), ops) in enumerate(zip(seqs, op_lists)):
        for v in (ops, split_runs(ops, rng), end_indels(ops), all_indels(len(a), len(b), k % 2 == 1)):
            sx.append(a)
            sy.append(b)
            cig.append(v)
    return sx, sy, cig


def job_cigars():
    """make_inputs' true alignments on the forward strand (the minus strands rebased, as job_prepare does)"""
    _, jobs = make_inputs(np.random.default_rng(61), 12, 300)
    return [(j["subX"], j["subY"]) for j in jobs], [j["ops"] for j in jobs]


def decoded_cigars(ctx, p):
    """PAIRS with the cigars of device chains and MEAs"""
    b = _batch(ctx, "device", p)
    try:
        b.run(_model(5), p, cp.MODE_ALIGNED_PAIRS_INDELS)
        out = []
        for decode in (lambda: b.ordered_chain(0.5), lambda: b.mea(p.gapGamma, left_shift=True)):
            decode()
            out += unpacked(b.alignment_cigars())
    finally:
        b.close()
    return [(q[1], q[2]) for q in PAIRS] * 2, out


def _check_anchors(ctx, host, keep, seqs, op_lists, seed, what):
    sx, sy, cig = variants(seqs, op_lists, seed)
    cigars = packed(cig)
    p = param_sets()["realign"]
    for trim in (0, 1, 3, BIG_TRIM):
        cols = [host_anchors(host, ops, a, b, trim, 0) for a, b, ops in zip(sx, sy, cig)]
        for expansion in (0, 10, 3):
            b = keep(cp.Batch.from_cigars(ctx, sx, sy, cigars, with_band(p, trim, expansion)))
            got = _per_pair(*b.fetch_anchors())
            for k, (g, c) in enumerate(zip(got, cols)):
                want = c.copy()
                want[:, 2] = expansion
                assert np.array_equal(g, want), "%s, pair %d (variant %d), trim %d, expansion %d: %d device anchors, %d host anchors" % (
                    what, k // 4, k % 4, trim, expansion, len(g), len(want))
            if trim == BIG_TRIM:
                assert b.fetch_anchors()[0][-1] == 0
            b.close()


def test_anchors_of_true_alignments_equal_the_hosts(ctx, host, keep):
    seqs, ops = job_cigars()
    _check_anchors(ctx, host, keep, seqs, ops, 1, "make_inputs")


def test_anchors_of_decoded_alignments_equal_the_hosts(ctx, host, keep):
    seqs, ops = decoded_cigars(ctx, param_sets()["realign"])
    assert sum(len(o) for o in ops) > 1000
    _check_anchors(ctx, host, keep, seqs, ops, 2, "PAIRS")


def test_empty_batch_and_empty_sequences(ctx, keep):
    p = param_sets()["realign"]
    b = keep(cp.Batch.from_cigars(ctx, [], [], packed([]), p))
    off, tri = b.fetch_anchors()
    assert off.tolist() == [0] and len(tri) == 0
    b = keep(cp.Batch.from_cigars(ctx, [b"", b"ACGT", b""], [b"", b"", b"ACG"], packed([[], [(cp.OP_INDEL_X, 4)], [(cp.OP_INDEL_Y, 3), (cp.OP_MATCH, 0)]]), p))
    assert b.fetch_anchors()[0].tolist() == [0, 0, 0, 0]


@pytest.mark.parametrize("which", ["realign", "em"])
def test_round_trip_equals_reanchoring(ctx, keep, which):
    """from_cigars of a batch's alignment cigars gives the anchors anchors_from_alignments gives for those alignments"""
    p = param_sets()[which]
    b = keep(_batch(ctx, "device", p))
    b.run(_model(5), p, cp.MODE_ALIGNED_PAIRS)
    b.reweight_pairs(p.gapGamma)
    b.ordered_chain(0.85)
    sx, sy = [q[1] for q in PAIRS], [q[2] for q in PAIRS]
    for trim, expansion in ((0, 10), (2, 4), (3, 3)):
        q = with_band(p, trim, expansion)
        cigars = b.alignment_cigars()
        c = keep(cp.Batch.from_cigars(ctx, sx, sy, cigars, q))
        b.anchors_from_alignments(q)
        want, got = b.fetch_anchors(), c.fetch_anchors()
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), "trim %d, expansion %d" % (trim, expansion)
        c.close()


@pytest.mark.parametrize("S", [5, 3])
def test_batch_from_cigars_runs_as_a_created_one(ctx, keep, S):
    p = param_sets()["realign"]
    sM = _model(S)
    seqs, ops = decoded_cigars(ctx, p)
    n = len(PAIRS)
    sx, sy = [q[1] for q in PAIRS], [q[2] for q in PAIRS]
    rl, rr = [q[3] for q in PAIRS], [q[4] for q in PAIRS]
    b = keep(cp.Batch.from_cigars(ctx, sx, sy, packed(ops[:n]), p, rl, rr))
    fresh = keep(_fresh(ctx, b))
    for mode in (cp.MODE_ALIGNED_PAIRS, cp.MODE_ALIGNED_PAIRS_INDELS, cp.MODE_EXPECTATIONS, cp.MODE_FORWARD):
        b.run(sM, p, mode)
        fresh.run(sM, p, mode)
        _assert_same_outputs(_outputs(b, mode), _outputs(fresh, mode), mode, "%d-state, mode %d" % (S, mode))
    # an odd expansion is refused by a dynamicAnchorExpansion run, as for a created batch with those anchors
    b = keep(cp.Batch.from_cigars(ctx, sx, sy, packed(ops[n:]), with_band(p, 1, 5), rl, rr))
    assert np.all(b.fetch_anchors()[1][:, 2] == 5)
    fresh = keep(_fresh(ctx, b))
    dyn = with_band(p, 0, 10)
    dyn.dynamicAnchorExpansion = 1
    for batch in (b, fresh):
        with pytest.raises(cp.CpbError, match="error 2: pair .*dynamicAnchorExpansion"):
            batch.run(sM, dyn, cp.MODE_ALIGNED_PAIRS)
    dyn.dynamicAnchorExpansion = 0
    b.run(sM, dyn, cp.MODE_ALIGNED_PAIRS)
    fresh.run(sM, dyn, cp.MODE_ALIGNED_PAIRS)
    _assert_same_outputs(_outputs(b, cp.MODE_ALIGNED_PAIRS), _outputs(fresh, cp.MODE_ALIGNED_PAIRS), cp.MODE_ALIGNED_PAIRS, "expansion 5")


# ---- weighing a cigar's columns against list 0 ----
def _check_weighed(host, b, sx, sy, op_lists, what, trims=(0, 1, 3)):
    cigars = packed(op_lists)
    lists = _per_pair(*b.fetch_pairs(0, reference_order=True))
    for trim in trims:
        b.alignments_from_cigars(cigars, trim)
        got = _per_pair(*b.fetch_alignments())
        scores = np.array([b.score_alignments(kind) for kind in range(4)]).T
        coff, cops = b.alignment_cigars()
        for k, (a, c, ops, l0, g) in enumerate(zip(sx, sy, op_lists, lists, got)):
            hosted = host_weighed(host_columns(host, ops, trim), l0)
            want = hosted[np.argsort(hosted[:, 1], kind="stable")]
            assert np.array_equal(g, want), "%s, trim %d, pair %d: %d device columns, %d host columns" % (what, trim, k, len(g), len(want))
            ws = host.scores(cp.binding._as_bytes(a).decode(), cp.binding._as_bytes(c).decode(), hosted)
            assert _same_bits(scores[k], ws), "%s, trim %d, pair %d: scores %s, host %s" % (what, trim, k, scores[k], ws)
            cols = [(int(t[1]), int(t[2])) for t in g]
            assert [tuple(o) for o in cops[coff[k]:coff[k + 1]].tolist()] == ops_from_columns(cols, len(a), len(c)), "%s, pair %d" % (what, k)


def test_weights_equal_the_hosts(ctx, host, keep):
    p = param_sets()["realign"]
    sM = _model(5)
    seqs, ops = decoded_cigars(ctx, p)
    sx, sy, cig = variants(seqs, ops, 3)
    b = keep(cp.Batch.from_cigars(ctx, sx, sy, packed(cig), p))
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)
    _check_weighed(host, b, sx, sy, cig, "raw")
    b.reweight_pairs(p.gapGamma)
    _check_weighed(host, b, sx, sy, cig, "reweighted")
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS_INDELS)
    _check_weighed(host, b, sx, sy, cig, "INDELS")


RESCORE = {None: None, "--rescoreByIdentity": cp.SCORE_IDENTITY, "--rescoreByPosteriorProb": cp.SCORE_POSTERIOR}


@pytest.mark.parametrize("option", sorted(RESCORE, key=str))
def test_flat_composition_is_the_programs_rescoring(tmp_path, ctx, keep, option):
    """cpb_batch_create_from_cigars with cPecanRealign's parameters, an ALIGNED_PAIRS run, cpb_batch_alignments_from_cigars at its trim,
    then scores and cigars: the lines cPecanRealign --rescoreOriginalAlignment prints, score text included"""
    fasta, jobs = make_inputs(np.random.default_rng(62), 8, 300)
    args = ["--rescoreOriginalAlignment"] + ([option] if option else [])
    got = run(tmp_path, fasta, jobs, args).stdout.splitlines()
    p = cli_params()
    cigars = packed([j["ops"] for j in jobs])
    b = keep(cp.Batch.from_cigars(ctx, [j["subX"] for j in jobs], [j["subY"] for j in jobs], cigars, p, [1] * len(jobs), [1] * len(jobs)))
    b.run(cp.stateMachine5_construct(), p, cp.MODE_ALIGNED_PAIRS)
    b.alignments_from_cigars(cigars, p.constraintDiagonalTrim)
    scores = b.score_alignments(RESCORE[option]) if option else np.ones(len(jobs))
    off, ops = b.alignment_cigars()
    want = []
    for k, j in enumerate(jobs):
        f = cigar_line(j["name1"], j["s1"], j["e1"], 1, j["name2"], j["s2"], j["e2"], j["strand2"], 0.0, ops[off[k]:off[k + 1]].tolist()).split(" ")
        f[9] = score_text(scores[k])
        want.append(" ".join(f))
    assert got == want


# ---- the rules of a decode call, and the errors ----
def test_decode_call_rules(ctx, keep):
    p = param_sets()["realign"]
    sM = _model(5)
    seqs, ops = job_cigars()
    cigars = packed(ops)
    b = keep(cp.Batch.from_cigars(ctx, [a for a, _ in seqs], [c for _, c in seqs], cigars, p))
    anchors = b.fetch_anchors()

    def refused(call):
        with pytest.raises(cp.CpbError, match="error 2: cpb_batch_alignments_from_cigars"):
            call()
        with pytest.raises(cp.CpbError, match="error 2: cpb_batch_fetch_alignments"):
            b.fetch_alignments()

    refused(lambda: b.alignments_from_cigars(cigars))  # no run yet
    for mode in (cp.MODE_EXPECTATIONS, cp.MODE_FORWARD):
        b.run(sM, p, mode)
        refused(lambda: b.alignments_from_cigars(cigars))
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)
    b.ordered_chain(0.85)
    b.alignment_cigars()
    b.alignments_from_cigars(cigars)  # replaces the chain, discards its cigars
    with pytest.raises(cp.CpbError, match="error 2: cpb_batch_fetch_cigars"):
        cp.binding._check(cp.lib.cpb_batch_fetch_cigars(b.h, None))
    want = b.fetch_alignments()
    assert unpacked(b.alignment_cigars()) == [[tuple(o) for o in j] for j in ops]  # the true alignments start and end with a column
    b.reweight_pairs(p.gapGamma)  # leaves the list
    got = b.fetch_alignments()
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    b.anchors_from_alignments(p)  # works on it as on a chain: the cigar is the input's, and so are the anchors
    got = b.fetch_anchors()
    assert np.array_equal(got[0], anchors[0]) and np.array_equal(got[1], anchors[1])
    refused(lambda: b.alignments_from_cigars(cigars, -1))  # a refused call leaves no list
    b.alignments_from_cigars(cigars)
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)  # a run clears it
    with pytest.raises(cp.CpbError, match="error 2: cpb_batch_fetch_alignments"):
        b.fetch_alignments()


def test_error_paths(ctx, keep):
    lib = cp.lib
    p = param_sets()["realign"]
    sx, sy = [b"ACGTACGT", b"", b"AC"], [b"ACGTAC", b"A", b""]
    good = [[(cp.OP_MATCH, 6), (cp.OP_INDEL_X, 2)], [(cp.OP_INDEL_Y, 1)], [(cp.OP_INDEL_X, 2)]]
    bx, xo = cp.binding._pack_sequences(sx)
    by, yo = cp.binding._pack_sequences(sy)

    def create(off, ops, params=p, xo=xo):
        h = C.c_void_p(12345)
        rc = lib.cpb_batch_create_from_cigars(ctx.h, len(sx), bx.ctypes.data, xo.ctypes.data if xo is not None else None, by.ctypes.data,
                                              yo.ctypes.data, off.ctypes.data if off is not None else None,
                                              ops.ctypes.data if ops is not None else None, None, None,
                                              C.byref(params) if params is not None else None, C.byref(h))
        if rc == 0:
            lib.cpb_batch_destroy(h)
        return rc, h.value

    def refused(off, ops, what, **kw):
        rc, h = create(off, ops, **kw)
        assert rc == 2 and h is None, what
        msg = lib.cpb_last_error().decode()
        assert msg.startswith("cpb_batch_create_from_cigars"), msg
        return msg

    off, ops = packed(good)
    assert create(off, ops)[0] == 0
    refused(off, ops, "no parameters", params=None)
    for field in ("constraintDiagonalTrim", "diagonalExpansion"):
        for v in (-1, 1 << 31):
            q = with_band(p, 0, 4)
            setattr(q, field, v)
            refused(off, ops, field, params=q)
    refused(None, ops, "no offsets")
    refused(off + 1, ops, "offsets not from 0")
    bad = off.copy()
    bad[1], bad[2] = 2, 1
    refused(bad, ops, "decreasing")
    refused(off, None, "ops NULL")
    for t, n in ((3, 1), (-1, 1), (cp.OP_MATCH, -1)):
        o = ops.copy()
        o[1] = (t, n)
        assert "pair 0" in refused(off, o, "operation (%d, %d)" % (t, n))
    o = ops.copy()
    o[0, 1] = 5
    assert "pair 0" in refused(off, o, "short walk")
    o = ops.copy()
    o[2] = (cp.OP_INDEL_Y, 2)
    assert "pair 1" in refused(off, o, "walk past the end")
    refused(off, ops, "sequence offsets", xo=xo[::-1].copy())

    # cpb_batch_alignments_from_cigars: the same checks against the batch's lengths
    b = keep(cp.Batch.from_cigars(ctx, sx, sy, (off, ops), p))
    b.run(_model(5), p, cp.MODE_ALIGNED_PAIRS)

    def refused2(call):
        with pytest.raises(cp.CpbError, match="error 2: cpb_batch_alignments_from_cigars"):
            call()

    refused2(lambda: cp.binding._check(lib.cpb_batch_alignments_from_cigars(b.h, None, ops.ctypes.data, 0)))
    refused2(lambda: b.alignments_from_cigars((off + 1, ops)))
    refused2(lambda: b.alignments_from_cigars((bad, ops)))
    refused2(lambda: cp.binding._check(lib.cpb_batch_alignments_from_cigars(b.h, off.ctypes.data, None, 0)))
    for t, n in ((3, 1), (cp.OP_MATCH, -1)):
        o = ops.copy()
        o[1] = (t, n)
        refused2(lambda: b.alignments_from_cigars((off, o)))
    o = ops.copy()
    o[0, 1] = 5
    refused2(lambda: b.alignments_from_cigars((off, o)))
    for trim in (-1, 1 << 31):
        refused2(lambda: b.alignments_from_cigars((off, ops), trim))
    b.alignments_from_cigars((off, ops))
    assert b.fetch_alignments()[0].tolist() == [0, 6, 6, 6]


def test_small_scratch_budget_gives_the_same_results(ctx, host, keep):
    p = param_sets()["realign"]
    seqs, ops = decoded_cigars(ctx, p)
    sx, sy = [a for a, _ in seqs], [c for _, c in seqs]
    cigars = packed(ops)

    def results():
        b = keep(cp.Batch.from_cigars(ctx, sx, sy, cigars, p))
        b.run(_model(5), p, cp.MODE_ALIGNED_PAIRS)
        b.alignments_from_cigars(cigars, 1)
        out = [b.fetch_anchors(), b.fetch_alignments(), b.alignment_cigars()]
        b.close()
        return out

    want = results()
    try:
        ctx.set_scratch_budget(1 << 20)
        got = results()
    finally:
        ctx.set_scratch_budget(0)
    for g, w in zip(got, want):
        assert np.array_equal(g[0], w[0]) and np.array_equal(g[1], w[1])


def test_two_thousand_kilobase_alignments(ctx, host, keep):
    _, jobs = make_inputs(np.random.default_rng(63), 2000, 1000)
    sx, sy, op_lists = [j["subX"] for j in jobs], [j["subY"] for j in jobs], [j["ops"] for j in jobs]
    cigars = packed(op_lists)
    p = cli_params()
    b = keep(cp.Batch.from_cigars(ctx, sx, sy, cigars, p))
    got = _per_pair(*b.fetch_anchors())
    for k, (a, c, ops) in enumerate(zip(sx, sy, op_lists)):
        assert np.array_equal(got[k], host_anchors(host, ops, a, c, 0, int(p.diagonalExpansion))), "pair %d" % k
    b.run(_model(5), p, cp.MODE_ALIGNED_PAIRS)
    lists = _per_pair(*b.fetch_pairs(0, reference_order=True))
    b.alignments_from_cigars(cigars, 0)
    weighed = _per_pair(*b.fetch_alignments())
    for k, ops in enumerate(op_lists):
        hosted = host_weighed(host_columns(host, ops, 0), lists[k])
        assert np.array_equal(weighed[k], hosted[np.argsort(hosted[:, 1], kind="stable")]), "pair %d" % k
