"""Re-anchoring a batch from its own alignments on the device (cpb_batch_anchors_from_alignments; k_reanchor_* of decode_kernels.cuh) and
cPecanEm --updateTheBand, which realigns and re-anchors between EM iterations (cpecanResidentBatch_updateAnchors).

The definition of the new anchors is what cPecanRealign and cPecanEm do on the host with an alignment: its cigar (pairs_to_alignment, here
ops_from_columns), convertPairwiseForwardStrandAlignmentToAnchorPairs of libcpecan.so, then job_prepare's columns_match filter.  Every
comparison of anchors is exact."""
import os
import subprocess

import numpy as np
import pytest

import cpecan_b200 as cp
import helpers
from test_gpu_alignments import PAIRS, _batch, _model, _per_pair, _same_bits, param_sets
from test_gpu_realign_cli import EM_EXE, cigar_line, em_params, make_inputs, ops_from_columns, read_model
from test_realign_host import Host, host_cigar_anchors

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def host():
    return Host()


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


def host_anchors(host, cols, sX, sY, trim, expansion):
    """job_prepare's anchors (host/realignJobs.h) of the alignment with these (x, y) columns over the whole of sX and sY"""
    ops = np.array(ops_from_columns([(int(x), int(y)) for x, y in cols], len(sX), len(sY)), dtype=np.int64).reshape(-1, 2)
    a = host_cigar_anchors(host, ops, 0, 0, trim, expansion)
    ux, uy = np.frombuffer(sX.upper(), dtype=np.uint8), np.frombuffer(sY.upper(), dtype=np.uint8)
    if len(a) == 0:
        return a.reshape(0, 3)
    cx, cy = ux[a[:, 0]], uy[a[:, 1]]
    return a[(cx == cy) & (cx != ord("N"))]


def with_band(p, trim, expansion):
    q = cp.CpbParams.from_buffer_copy(p)
    q.constraintDiagonalTrim, q.diagonalExpansion = trim, expansion
    return q


def _check_lists(host, b, p, what):
    alns = _per_pair(*b.fetch_alignments())
    for trim in (0, 1, 3):
        for expansion in (0, 10):
            b.anchors_from_alignments(with_band(p, trim, expansion))
            got = _per_pair(*b.fetch_anchors())
            for q, aln, g in zip(PAIRS, alns, got):
                want = host_anchors(host, aln[:, 1:], q[1], q[2], trim, expansion)
                assert np.array_equal(g, want), "%s, trim %d, expansion %d, %s: %d device anchors, %d host anchors" % (
                    what, trim, expansion, q[0], len(g), len(want))


SETUPS = [(S, which) for S in (5, 3) for which in ("defaults", "realign", "em")]


@pytest.mark.parametrize("S,which", SETUPS)
def test_anchors_equal_the_hosts(ctx, host, keep, S, which):
    p = param_sets()[which]
    sM = _model(S)
    b = keep(_batch(ctx, "device", p))
    what = "%d-state, %s parameters" % (S, which)
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS_INDELS)
    for gamma in (0.5, 0.85):
        b.ordered_chain(gamma)
        _check_lists(host, b, p, what + ", chain %g" % gamma)
    for shift in (False, True):
        b.mea(p.gapGamma, left_shift=shift)
        _check_lists(host, b, p, what + ", MEA%s" % (" shifted" if shift else ""))
    b.reweight_pairs(p.gapGamma)
    b.ordered_chain(0.85)
    _check_lists(host, b, p, what + ", reweighted chain")
    b.close()


def _outputs(b, mode):
    if mode == cp.MODE_ALIGNED_PAIRS:
        return [b.fetch_pairs(0)]
    if mode == cp.MODE_ALIGNED_PAIRS_INDELS:
        return [b.fetch_pairs(k) for k in range(3)]
    if mode == cp.MODE_EXPECTATIONS:
        return list(b.fetch_expectations(per_pair=True))
    return [b.fetch_forward()]


def _assert_same_outputs(got, want, mode, what):
    for g, w in zip(got, want):
        if mode == cp.MODE_EXPECTATIONS:
            np.testing.assert_allclose(g, w, rtol=1e-9, err_msg=what)  # DESIGN §3
        elif isinstance(g, tuple):
            assert np.array_equal(g[0], w[0]) and np.array_equal(g[1], w[1]), what
        else:
            assert _same_bits(g, w), what


def _fresh(ctx, b, pairs=PAIRS):
    """a batch cpb_batch_create builds from the anchors b holds"""
    off, tri = b.fetch_anchors()
    return cp.Batch(ctx, [q[1] for q in pairs], [q[2] for q in pairs], [tri[off[i]:off[i + 1]] for i in range(len(pairs))],
                    [q[3] for q in pairs], [q[4] for q in pairs])


@pytest.mark.parametrize("S", [5, 3])
def test_reanchored_batch_runs_as_a_created_one(ctx, keep, S, monkeypatch):
    monkeypatch.delenv("CPB_NO_PLAN_CACHE", raising=False)
    p = param_sets()["em"]
    sM = _model(S)
    b = keep(_batch(ctx, "device", p))
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)
    assert b.stats().planReused == 1  # the plan cache is on
    before = b.fetch_anchors()
    b.reweight_pairs(p.gapGamma)
    b.ordered_chain(0.85)
    b.anchors_from_alignments(p)
    after = b.fetch_anchors()
    assert not (np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1]))  # the band moved
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)  # same mode, same parameters: planned anew all the same
    assert b.stats().planReused == 0
    fresh = keep(_fresh(ctx, b))
    for mode in (cp.MODE_ALIGNED_PAIRS, cp.MODE_ALIGNED_PAIRS_INDELS, cp.MODE_EXPECTATIONS, cp.MODE_FORWARD):
        b.run(sM, p, mode)
        fresh.run(sM, p, mode)
        _assert_same_outputs(_outputs(b, mode), _outputs(fresh, mode), mode, "%d-state, mode %d" % (S, mode))
    # anchors of an odd expansion: a dynamicAnchorExpansion run (whose own diagonalExpansion is even, as every run's must be) is refused,
    # as for a created batch with those anchors; a static run is not
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)
    b.ordered_chain(0.85)
    b.anchors_from_alignments(with_band(p, 0, 5))
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


def test_last_run_results_survive(ctx, keep):
    p = param_sets()["defaults"]
    b = keep(_batch(ctx, "device", p))
    b.run(_model(5), p, cp.MODE_ALIGNED_PAIRS_INDELS)
    b.reweight_pairs(p.gapGamma)
    b.ordered_chain(0.85)

    def snapshot():
        return ([b.fetch_pairs(k) for k in range(3)] + [b.fetch_pairs(k, reference_order=True) for k in range(3)] + [b.fetch_alignments()],
                [b.score_alignments(kind) for kind in range(4)], b.stats().reweighted)

    lists, scores, reweighted = snapshot()
    b.anchors_from_alignments(with_band(p, 2, 10))
    lists2, scores2, reweighted2 = snapshot()
    assert reweighted == reweighted2 == 1
    for g, w in zip(lists2, lists):
        assert np.array_equal(g[0], w[0]) and np.array_equal(g[1], w[1])
    for g, w in zip(scores2, scores):
        assert _same_bits(g, w)
    b.close()


def test_small_scratch_budget_gives_the_same_anchors(ctx, keep):
    p = param_sets()["em"]
    b = keep(_batch(ctx, "device", p))
    b.run(_model(5), p, cp.MODE_ALIGNED_PAIRS)
    b.ordered_chain(0.85)
    try:
        b.anchors_from_alignments(p)
        want = b.fetch_anchors()
        ctx.set_scratch_budget(1 << 16)  # a few pairs per chunk
        b.anchors_from_alignments(with_band(p, 3, 2))
        b.anchors_from_alignments(p)
        got = b.fetch_anchors()
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    finally:
        ctx.set_scratch_budget(0)
    b.close()


def test_error_paths_leave_the_batch_as_it_was(ctx, keep):
    p = param_sets()["em"]
    sM = _model(5)
    pairs = [q for q in PAIRS if q[0] in ("evolved12000_0", "tandem", "iupac_mixed", "empty_y")]
    b = keep(_batch(ctx, "device", p, pairs))
    anchors = b.fetch_anchors()
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)
    outputs = _outputs(b, cp.MODE_ALIGNED_PAIRS)

    def refused(call, code=2):
        with pytest.raises(cp.CpbError, match="error %d: cpb_batch_anchors_from_alignments" % code):
            call()
        got = b.fetch_anchors()
        assert np.array_equal(got[0], anchors[0]) and np.array_equal(got[1], anchors[1])

    refused(lambda: b.anchors_from_alignments(p))  # no decode yet
    b.ordered_chain(0.85)
    refused(lambda: b.anchors_from_alignments(None))
    for field in ("constraintDiagonalTrim", "diagonalExpansion"):
        for v in (-1, 1 << 31, 1 << 40):
            q = with_band(p, 0, 10)
            setattr(q, field, v)
            refused(lambda: b.anchors_from_alignments(q))
    ctx.set_scratch_budget(8192)  # less than the 12 kb pair's work array
    try:
        refused(lambda: b.anchors_from_alignments(p), code=5)
    finally:
        ctx.set_scratch_budget(0)
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)  # the run cleared the alignment list
    _assert_same_outputs(_outputs(b, cp.MODE_ALIGNED_PAIRS), outputs, cp.MODE_ALIGNED_PAIRS, "after the refusals")
    refused(lambda: b.anchors_from_alignments(p))
    b.run(sM, p, cp.MODE_EXPECTATIONS)
    refused(lambda: b.anchors_from_alignments(p))
    b.run(sM, p, cp.MODE_ALIGNED_PAIRS)
    _assert_same_outputs(_outputs(b, cp.MODE_ALIGNED_PAIRS), outputs, cp.MODE_ALIGNED_PAIRS, "after the refusals")
    b.close()


# ---- cPecanEm --updateTheBand ----
def perturbed_inputs(seed, n, length):
    """make_inputs' alignments with the columns of their middle half moved 3 positions along Y: the band of the input cigars is off"""
    fasta, jobs = make_inputs(np.random.default_rng(seed), n, length)
    for j in jobs:
        lY, cols = len(j["subY"]), j["cols"]
        lo, hi = len(cols) // 4, 3 * len(cols) // 4
        moved, py = [], -1
        for k, (x, y) in enumerate(cols):
            y = y + 3 if lo <= k < hi else y
            if py < y < lY:
                moved.append((x, y))
                py = y
        j["cols"] = moved
        j["ops"] = ops_from_columns(moved, len(j["subX"]), lY)
    return fasta, jobs


def run_em(tmp_path, fasta, jobs, args, env=None):
    fa = tmp_path / "seqs.fa"
    fa.write_text("".join("%s\n%s\n" % (h, s) for h, s in fasta))
    cig = "".join(cigar_line(j["name1"], j["s1"], j["e1"], 1, j["name2"], j["s2"], j["e2"], j["strand2"], 1.0, j["ops"]) + "\n" for j in jobs)
    out = subprocess.run([EM_EXE] + args + [str(fa)], input=cig, capture_output=True, text=True, env=env)
    assert out.returncode == 0, out.stderr


@pytest.mark.parametrize("trim", [0, 2])
@pytest.mark.parametrize("type_,name", [(cp.fiveState, "fiveState"), (cp.threeState, "threeState")])
def test_em_update_the_band_matches_the_oracle(tmp_path, host, type_, name, trim):
    """three iterations, emissions trained; after iterations 1 and 2 the oracle's aligned pairs under the new model, reweighted, chained at
    matchGamma 0.85 and turned into anchors, as cPecanRealign --loadHmm would realign them and cPecanEm read them back"""
    from cpecan_b200 import sharding

    oracle = helpers.best_oracle()
    fasta, jobs = perturbed_inputs(48, 10, 250)
    args = ["--iterations", "3", "--trainEmissions", "--modelType", name, "--constraintDiagonalTrim", str(trim)]
    run_em(tmp_path, fasta, jobs, args + ["--updateTheBand", "--outputModel", str(tmp_path / "band.hmm")])
    run_em(tmp_path, fasta, jobs, args + ["--outputModel", str(tmp_path / "fixed.hmm")])
    got, fixed = read_model(tmp_path / "band.hmm"), read_model(tmp_path / "fixed.hmm")
    S = 5 if type_ == cp.fiveState else 3
    p = em_params()
    p.constraintDiagonalTrim = trim
    op = helpers.orc_params_from(p)
    anchors = [host_anchors(host, j["cols"], j["subX"].encode(), j["subY"].encode(), trim, 10) for j in jobs]
    trans, emis, running = np.full(S * S, 1.0 / S), np.full(S * 16, 1.0 / 16), []
    for it in range(3):
        spec = helpers.ModelSpec(type_, trans.reshape(S, S), emis.reshape(S, 16))
        total = np.zeros(cp.hmm_len(S))
        for j, a in zip(jobs, anchors):
            total += oracle.expectations(spec.orc(), op, j["subX"], j["subY"], a, True, True)
        total[:-1] += 1e-12
        running.append(total[-1])
        hmm = sharding.normalise_hmm(total, S)
        trans, emis = hmm[:S * S], hmm[S * S:S * S + 16 * S]
        if it < 2:
            spec = helpers.ModelSpec(type_, trans.reshape(S, S), emis.reshape(S, 16))
            for k, j in enumerate(jobs):
                sX, sY = j["subX"], j["subY"]
                pairs = oracle.aligned_pairs(spec.orc(), op, sX, sY, anchors[k], True, True)
                chain = host.chain(host.reweight(pairs, len(sX), len(sY), float(p.gapGamma)), sX, sY, 0.85)
                anchors[k] = host_anchors(host, chain[:, 1:], sX.encode(), sY.encode(), trim, 10)
    np.testing.assert_allclose(got["transitions"], trans, rtol=1e-7, atol=1e-12)
    np.testing.assert_allclose(got["emissions"], emis, rtol=1e-7, atol=1e-12)
    np.testing.assert_allclose(got["running"], running, rtol=1e-9)
    np.testing.assert_allclose(got["running"][0], fixed["running"][0], rtol=1e-9)  # the first iteration runs in the input alignments' band
    assert all(abs(g - f) > 1e-9 * abs(f) for g, f in zip(got["running"][1:], fixed["running"][1:]))  # then the band moved


def test_em_update_the_band_needs_two_iterations(tmp_path):
    fasta, jobs = perturbed_inputs(49, 6, 200)
    for flags, out in (([], "a.hmm"), (["--updateTheBand"], "b.hmm")):
        run_em(tmp_path, fasta, jobs, ["--iterations", "1", "--randomStart", "--trials", "2", "--seed", "11", "--outputModel", str(tmp_path / out)] + flags)
    assert (tmp_path / "a.hmm").read_bytes() == (tmp_path / "b.hmm").read_bytes()


def test_em_update_the_band_on_two_contexts(tmp_path):
    """two engine contexts on one GPU ($CPECAN_DEVICE_LIST=0,0): each re-anchors its share of the alignments"""
    fasta, jobs = perturbed_inputs(50, 10, 250)
    args = ["--iterations", "3", "--trainEmissions", "--updateTheBand", "--randomStart", "--trials", "2", "--seed", "3"]
    env = dict(os.environ)
    env.pop("CPECAN_DEVICE_LIST", None)
    env.pop("CPECAN_DEVICES", None)
    run_em(tmp_path, fasta, jobs, args + ["--outputModel", str(tmp_path / "one.hmm")], env)
    env["CPECAN_DEVICE_LIST"] = "0,0"
    run_em(tmp_path, fasta, jobs, args + ["--outputModel", str(tmp_path / "two.hmm")], env)
    one, two = read_model(tmp_path / "one.hmm"), read_model(tmp_path / "two.hmm")
    for key in ("transitions", "emissions", "running"):
        np.testing.assert_allclose(two[key], one[key], rtol=1e-9)
