"""cPecanRealign's realignment decoded on the device (getRealignedCigarsUsingAnchorsBatch of libcpecan.so: reweighting, ordered chain,
scores and cigar operations on the GPU) against the pipeline of tests/test_gpu_realign_cli.py: the oracle's aligned pairs, then the host
list functions, then the cigar, compared line for line including the score text.  The posterior files are compared with what the host
route writes from the device's own posteriors."""
import math
import os
import subprocess

import numpy as np
import pytest

import cpecan_b200 as cp
import helpers
from test_gpu_realign_cli import EXE, cigar_line, cli_params, expected_line, make_inputs
from test_realign_host import Host

pytestmark = pytest.mark.gpu

MINUS_STRAND_JOBS = 3  # make_inputs puts sequence 2 of every odd alignment on the minus strand


@pytest.fixture(scope="module")
def inputs():
    return make_inputs(np.random.default_rng(50), 2 * MINUS_STRAND_JOBS, 300)


@pytest.fixture(scope="module")
def host():
    return Host()


def run(tmp_path, fasta, jobs, args, env=None):
    fa = tmp_path / "seqs.fa"
    fa.write_text("".join("%s\n%s\n" % (h, s) for h, s in fasta))
    cig = "".join(cigar_line(j["name1"], j["s1"], j["e1"], 1, j["name2"], j["s2"], j["e2"], j["strand2"], 1.0, j["ops"]) + "\n" for j in jobs)
    out = subprocess.run([EXE] + args + [str(fa)], input=cig, capture_output=True, text=True, env=env)
    assert out.returncode == 0, out.stderr
    return out


def score_text(v):
    """printf's %f: glibc writes a NaN with its sign"""
    if math.isnan(v):
        return "-nan" if math.copysign(1.0, v) < 0 else "nan"
    return "%f" % v


def anchors_of(job, expansion):
    sX, sY = job["subX"], job["subY"]
    return np.array([(x, y, expansion) for x, y in job["cols"] if sX[x].upper() == sY[y].upper() and sX[x].upper() != "N"],
                    dtype=np.int64).reshape(-1, 3)


def expected(oracle, host, jobs, spec=None, match_gamma=0.85, gap_gamma=0.5, kind=None):
    """the cigar line of every job as the host route writes it from the oracle's posteriors"""
    p = cli_params()
    p.gapGamma = gap_gamma
    spec = spec or helpers.ModelSpec(cp.fiveState)
    lines = []
    for j in jobs:
        sX, sY = j["subX"], j["subY"]
        pairs = oracle.aligned_pairs(spec.orc(), helpers.orc_params_from(p), sX, sY, anchors_of(j, int(p.diagonalExpansion)), True, True)
        chain = host.chain(host.reweight(pairs, len(sX), len(sY), gap_gamma), sX, sY, match_gamma)
        score = 1.0 if kind is None else host.scores(sX, sY, chain)[kind]
        f = expected_line(j, 0.0, [(int(t[1]), int(t[2])) for t in chain]).split(" ")
        f[9] = score_text(score)
        lines.append(" ".join(f))
    return lines


KINDS = {"--rescoreByIdentity": cp.SCORE_IDENTITY, "--rescoreByIdentityIgnoringGaps": cp.SCORE_IDENTITY_IGNORING_GAPS,
         "--rescoreByPosteriorProb": cp.SCORE_POSTERIOR, "--rescoreByPosteriorProbIgnoringGaps": cp.SCORE_POSTERIOR_IGNORING_GAPS}


@pytest.mark.parametrize("option", sorted(KINDS))
def test_rescore_options(tmp_path, inputs, host, option):
    fasta, jobs = inputs
    got = run(tmp_path, fasta, jobs, [option]).stdout.splitlines()
    assert got == expected(helpers.best_oracle(), host, jobs, kind=KINDS[option])


@pytest.mark.parametrize("args,match_gamma,gap_gamma,kind", [
    (["--matchGamma", "0"], 0.0, 0.5, None),
    (["--matchGamma", "1", "--rescoreByPosteriorProb"], 1.0, 0.5, cp.SCORE_POSTERIOR),
    (["--matchGamma", "1.5"], 1.5, 0.5, None),  # no pair qualifies: every alignment is all indels
    (["--matchGamma", "1.5", "--rescoreByIdentityIgnoringGaps"], 1.5, 0.5, cp.SCORE_IDENTITY_IGNORING_GAPS),
    (["--matchGamma", "1.5", "--rescoreByPosteriorProb"], 1.5, 0.5, cp.SCORE_POSTERIOR),
    (["--gapGamma", "0", "--rescoreByIdentity"], 0.85, 0.0, cp.SCORE_IDENTITY),
    (["--batchBases", "1500", "--rescoreByPosteriorProbIgnoringGaps"], 0.85, 0.5, cp.SCORE_POSTERIOR_IGNORING_GAPS),  # several passes
])
def test_gammas_and_passes(tmp_path, inputs, host, args, match_gamma, gap_gamma, kind):
    fasta, jobs = inputs
    got = run(tmp_path, fasta, jobs, args).stdout.splitlines()
    assert got == expected(helpers.best_oracle(), host, jobs, match_gamma=match_gamma, gap_gamma=gap_gamma, kind=kind)
    if match_gamma > 1:
        assert all(line.split()[10] != "M" and "M" not in line.split()[10::2] for line in got)


def test_load_three_state_hmm(tmp_path, inputs, host):
    fasta, jobs = inputs
    spec = helpers.ModelSpec(cp.threeState, [[0.90, 0.05, 0.05], [0.70, 0.28, 0.02], [0.70, 0.02, 0.28]],
                             np.vstack([np.full(16, 0.02) + np.eye(4).ravel() * 0.17, np.full(16, 0.0625), np.full(16, 0.0625)]))
    model = tmp_path / "three.hmm"
    model.write_text("%d %s 0.0\n%s\n" % (cp.threeState, " ".join("%.17g" % v for v in spec.transitions.ravel()),
                                           " ".join("%.17g" % v for v in spec.emissions.ravel())))
    got = run(tmp_path, fasta, jobs, ["--loadHmm", str(model), "--rescoreByPosteriorProb"]).stdout.splitlines()
    assert got == expected(helpers.best_oracle(), host, jobs, spec=spec, kind=cp.SCORE_POSTERIOR)


def test_posterior_files_and_split(tmp_path, ctx, inputs, host):
    """--outputPosteriorProbs / --outputAllPosteriorProbs hold the last alignment's chain / posteriors (rewritten per alignment), in
    original coordinates, in the order the host route writes them: posteriors in the reference's list order, the chain as it comes"""
    fasta, jobs = inputs
    probs, all_probs = tmp_path / "probs.tsv", tmp_path / "all.tsv"
    got = run(tmp_path, fasta, jobs, ["--outputPosteriorProbs", str(probs), "--outputAllPosteriorProbs", str(all_probs)]).stdout.splitlines()
    assert got == expected(helpers.best_oracle(), host, jobs)
    split = run(tmp_path, fasta, jobs, ["--splitIndelsLongerThanThis", "1"]).stdout.splitlines()
    assert len(split) > len(got)
    for line in split:
        ops = line.split()[10:]
        assert ops[0] == "M" and ops[-2] == "M"
    # the host route's files, from the device's posteriors of the last alignment
    j = jobs[-1]
    p = cli_params()
    sX, sY = j["subX"], j["subY"]
    b = cp.Batch(ctx, [sX.encode()], [sY.encode()], [anchors_of(j, int(p.diagonalExpansion))], [1], [1])
    b.run(cp.stateMachine5_construct(), p, cp.MODE_ALIGNED_PAIRS)
    _, raw = b.fetch_pairs(0, reference_order=True)
    b.close()
    chain = host.chain(host.reweight(raw.astype(np.int64), len(sX), len(sY), 0.5), sX, sY, 0.85)
    lo2, hi2 = min(j["s2"], j["e2"]), max(j["s2"], j["e2"])

    def rows(triples):
        return "".join("%d\t%d\t%f\n" % (j["s1"] + t[1], (lo2 + t[2]) if j["strand2"] else (hi2 - 1 - t[2]), t[0] / cp.PAIR_ALIGNMENT_PROB_1)
                       for t in np.asarray(triples, dtype=np.int64).reshape(-1, 3))

    assert not j["strand2"]  # the last job is on the minus strand: its coordinates are flipped
    assert all_probs.read_text() == rows(raw)
    assert probs.read_text() == rows(chain)


def test_the_cloud_stays_on_the_device(tmp_path, inputs):
    fasta, jobs = inputs
    env = dict(os.environ, CPECAN_HOST_TIMING="1")
    new = run(tmp_path, fasta, jobs, [], env=env).stderr
    assert "cigar operations" in new and "copy + reference order of" not in new
    old = run(tmp_path, fasta, jobs, ["--rescoreOriginalAlignment"], env=env).stderr  # the one route that still takes the posteriors
    assert "copy + reference order of" in old


def test_two_gpus(tmp_path, inputs, host):
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    fasta, jobs = inputs
    got = run(tmp_path, fasta, jobs, ["--gpus", "2", "--rescoreByIdentity"]).stdout.splitlines()
    assert got == expected(helpers.best_oracle(), host, jobs, kind=cp.SCORE_IDENTITY)
