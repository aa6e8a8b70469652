"""libcpecan.so -- the reference-named C API (include/cpecan/*.h) in plain C over the engine's C-ABI.

CPU part: the library exports every function the headers declare, and the host-only pieces (containers, Hmm text /
JSON formats, parameter JSON, split points, diagonals, symbols) pass tests/c/test_cpecan_api.c's `host` suite, which
restates the reference's own unit tests for them.  GPU part: the `gpu` suite (the reference's known-answer tests) and a
differential run of the C entry points -- batched and one-pair -- against the oracle.
"""
import os
import re
import subprocess

import numpy as np
import pytest

import helpers

ROOT = helpers.ROOT
LIB_DIR = os.path.join(ROOT, "cpecan_b200", "lib")
HOST_SO = os.path.join(LIB_DIR, "libcpecan.so")
BUILD = os.path.join(ROOT, "tests", "c", "_build")
EXE = os.path.join(BUILD, "test_cpecan_api")


PINT_TOL = 0  # integer output is bit-exact


def build_exe():
    src = os.path.join(ROOT, "tests", "c", "test_cpecan_api.c")
    if not os.path.exists(HOST_SO):
        subprocess.check_call(["make", "-s", "-f", os.path.join(ROOT, "cpecan_b200", "csrc", "Makefile")])
    if not os.path.exists(EXE) or os.path.getmtime(EXE) < max(os.path.getmtime(src), os.path.getmtime(HOST_SO)):
        os.makedirs(BUILD, exist_ok=True)
        subprocess.check_call(["gcc", "-std=c99", "-O1", "-D_POSIX_C_SOURCE=200809L", "-I" + os.path.join(ROOT, "include"), src, "-o", EXE,
                               "-L" + LIB_DIR, "-lcpecan", "-lcpecan_b200", "-Wl,-rpath," + LIB_DIR, "-lm"])
    return EXE


def declared_functions(header):
    text = open(header).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"typedef[^;]*\(\*\w+\)\([^;]*;", "", text)       # function-pointer typedefs
    text = re.sub(r"struct\s+\w+\s*\{.*?\};", "", text, flags=re.S)  # struct bodies (callback members)
    return sorted(set(re.findall(r"\b(\w+)\s*\([^;{}]*\)\s*;", text)) - {"defined"})


def test_host_library_exports_every_declared_symbol():
    build_exe()
    out = subprocess.check_output(["nm", "-D", "--defined-only", HOST_SO], text=True)
    exported = {line.split()[-1] for line in out.splitlines() if line.strip()}
    for h in ("sonLibLite.h", "stateMachine.h", "pairwiseAligner.h", "pairwiseAlignment.h", "multipleAligner.h"):
        names = declared_functions(os.path.join(ROOT, "include", "cpecan", h))
        assert len(names) > (0 if h == "multipleAligner.h" else 10), h
        missing = [n for n in names if n not in exported]
        assert not missing, "%s declares functions libcpecan.so does not export: %s" % (h, missing)


def test_host_library_has_no_dp_of_its_own():
    """The C host layer marshals; the recurrence lives only in the CUDA engine (no logAdd / cell update on the host)."""
    host_dir = os.path.join(ROOT, "cpecan_b200", "csrc", "host")
    for fn in os.listdir(host_dir):
        text = open(os.path.join(host_dir, fn)).read()
        assert "oracle" not in text.lower().replace("oracle/", "") or fn.endswith(".md")
        if fn == "cPecanEm.c":
            # the EM trainer's Jukes-Cantor starting emissions (cPecanEm.py:87-93) are the one exponential on the host side
            assert len(re.findall(r"\bexp\s*\(", text)) == 1 and "jukes_cantor_emissions" in text
            text = re.sub(r"\bexp\s*\(-4\.0 \* divergence / 3\.0\)", "", text)
        if fn == "logAdd.c":
            # the reference's header exposes logAdd (inc/pairwiseAligner.h:167); this file is that scalar and nothing else, and no
            # other host file may call it
            assert "cubic" in text and len(text.splitlines()) < 40
            continue
        assert not re.search(r"\blogAdd\s*\(|\bexp\s*\(|\blog\s*\(", text), fn


def test_host_logadd_is_bit_identical_to_the_reference(oracle):
    """logAdd (inc/pairwiseAligner.h:167) of libcpecan.so against the reference's own, over every segment, the cut-off and LOG_ZERO"""
    import ctypes as C

    build_exe()
    lib = C.CDLL(HOST_SO)
    lib.logAdd.restype = C.c_double
    lib.logAdd.argtypes = [C.c_double, C.c_double]
    rng = np.random.default_rng(7)
    xs = rng.uniform(-50, 5, 20000)
    ds = np.concatenate([rng.uniform(0, 9, 19000), [0.0, 1.0, 2.5, 4.5, 7.5, np.nextafter(1.0, 2), np.nextafter(7.5, 0)], rng.uniform(0, 1e-6, 993)])
    for x, d in zip(xs, ds):
        for u, v in ((x, x + d), (x + d, x)):
            assert lib.logAdd(u, v) == oracle.logadd(u, v), (u, v)
    inf = float("inf")
    for u, v in ((-inf, 1.5), (1.5, -inf), (-inf, -inf)):
        assert lib.logAdd(u, v) == oracle.logadd(u, v)


def test_host_suite_without_a_gpu():
    out = subprocess.run([build_exe(), "host"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert re.search(r"\d+ checks, 0 failures", out.stdout)


def test_alignment_entry_points_abort_loudly_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("needs a box without a GPU")
    out = subprocess.run([build_exe(), "gpu"], capture_output=True, text=True)
    assert out.returncode != 0
    assert "no CPU implementation" in out.stderr or "CUDA" in out.stderr


@pytest.mark.gpu
def test_reference_known_answer_tests_through_the_c_api():
    out = subprocess.run([build_exe(), "gpu"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert re.search(r"\d+ checks, 0 failures", out.stdout)


def _parse_list(fields):
    n = int(fields[0])
    return np.asarray([int(v) for v in fields[1:1 + 3 * n]], dtype=np.int64).reshape(-1, 3)


@pytest.mark.gpu
@pytest.mark.parametrize("type_, devices", [(0, None), (1, None), (2, None), (3, None), (0, "0,0"), (3, "0,0,0"), (0, "0,1"), (2, "0,1")])
def test_c_api_matches_the_oracle(tmp_path, oracle, type_, devices):
    """devices: $CPECAN_DEVICE_LIST -- "0,0" deals every batch over two engine contexts (here both on GPU 0): one host thread per
    context, problems dealt longest first, results back at their own indices, expectation totals summed across the contexts"""
    import cpecan_b200 as cp
    from cpecan_b200 import synth

    rng = np.random.default_rng(100 + type_)
    S = 5 if type_ < 2 else 3
    spec = helpers.ModelSpec.random(rng, type_) if type_ % 2 else helpers.ModelSpec(type_)
    hmm_file = "-"
    if spec.transitions is not None:
        hmm_file = str(tmp_path / "model.hmm")
        with open(hmm_file, "w") as f:  # the reference's text format with full precision (%f would round the model)
            f.write("%d\t%s\t0.0\n" % (type_, "\t".join(repr(float(v)) for v in spec.transitions.ravel())))
            f.write("\t".join(repr(float(v)) for v in spec.emissions.ravel()) + "\t\n")
    p = cp.pairwiseAlignmentBandingParameters_construct()
    p.minDiagsBetweenTraceBack = 60
    p.traceBackDiagonals = 10
    p.diagonalExpansion = 6
    p.splitMatrixBiggerThanThis = 400
    p.threshold = 0.05
    pj = ('{"threshold": %r, "minDiagsBetweenTraceBack": %d, "traceBackDiagonals": %d, "diagonalExpansion": %d, '
          '"splitMatrixBiggerThanThis": %d}' % (p.threshold, p.minDiagsBetweenTraceBack, p.traceBackDiagonals, p.diagonalExpansion,
                                                p.splitMatrixBiggerThanThis))
    packed = synth.evolved_pairs(6, 180, seed=41 + type_, trim=2, expansion=int(p.diagonalExpansion))
    cases = []
    for i in range(6):
        sx, sy, a = synth.unpack(packed, i)
        cases.append((sx, sy, np.asarray(a, dtype=np.int64).reshape(-1, 3), bool(i & 1), bool(i & 2)))
    cases.append(("ACGTN", "", np.zeros((0, 3), dtype=np.int64), False, False))  # an empty sequence
    cases.append(("acgtnACGT", "ACGTTACGT", np.zeros((0, 3), dtype=np.int64), True, True))
    inp, outp = tmp_path / "in.txt", tmp_path / "out.txt"
    with open(inp, "w") as f:
        f.write("%d %s %s\n%d\n" % (type_, hmm_file, pj, len(cases)))
        for sx, sy, a, rl, rr in cases:
            sx = sx if isinstance(sx, str) else bytes(sx).decode()
            sy = sy if isinstance(sy, str) else bytes(sy).decode()
            f.write("%d %d %d\n%s\n%s\n%s\n" % (rl, rr, a.shape[0], sx or "-", sy or "-", " ".join(str(int(v)) for v in a.ravel())))
    two_gpus = devices is not None and len(set(devices.split(","))) > 1
    if two_gpus:
        import torch

        if torch.cuda.device_count() < 2:
            pytest.skip("needs two GPUs")
    env = dict(os.environ)
    env.pop("CPECAN_DEVICE_LIST", None)
    if devices is not None:
        env["CPECAN_DEVICE_LIST"] = devices
    out = subprocess.run([build_exe(), "run", str(inp), str(outp)], capture_output=True, text=True, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    if devices is not None and not two_gpus:
        assert "summing the expectation totals" in out.stderr  # NCCL needs distinct GPUs: two contexts on one GPU take the host sum
    if two_gpus:
        assert "summing the expectation totals" not in out.stderr  # distinct GPUs: ncclAllReduce of the 58 / 106 doubles
    lines = open(outp).read().splitlines()
    om, op = spec.orc(), helpers.orc_params_from(p)
    total = np.zeros(cp.hmm_len(S))
    k = 0
    for i, (sx, sy, a, rl, rr) in enumerate(cases):
        assert lines[k] == "problem %d" % i
        got = {}
        for j in range(1, 19):
            f = lines[k + j].split()
            got[f[0]] = f[1:]
        k += 19
        want = oracle.aligned_pairs_with_indels(om, op, sx, sy, a, rl, rr)
        for key, w in zip(("match", "gapX", "gapY"), want):
            g, w = helpers.sort_triples(_parse_list(got[key])), helpers.sort_triples(w)
            assert g.shape == w.shape and np.array_equal(g[:, 1:], w[:, 1:]), (i, key)
            assert g.shape[0] == 0 or np.abs(g[:, 0] - w[:, 0]).max() <= PINT_TOL
        for key in ("only", "one"):
            g = helpers.sort_triples(_parse_list(got[key]))
            assert np.array_equal(g[:, 1:], helpers.sort_triples(want[0])[:, 1:]), (i, key)
        fw = oracle.forward_prob(om, op, sx, sy, a, rl, rr)
        assert float.fromhex(got["forward"][0]) == fw and float.fromhex(got["forward1"][0]) == fw
        e = oracle.expectations(om, op, sx, sy, a, rl, rr)
        np.testing.assert_allclose(np.array([float.fromhex(v) for v in got["expectations"]]), e, rtol=1e-9, atol=1e-12)
        total += e
        # the callback entry points (inc/pairwiseAligner.h:245, :264) with the three built-in callbacks.  Split form + the reference's
        # correction functions = the wrapper's list, element for element; the one-region form = the oracle without splitting, in the
        # callback's own order (the reverse of the wrapper's)
        for key, ref in (("splitting", "one"), ("splittingM", "match"), ("splittingX", "gapX"), ("splittingY", "gapY")):
            assert got[key] == got[ref], (i, key)
        np.testing.assert_allclose(np.array([float.fromhex(v) for v in got["splittingE"]]), e, rtol=1e-9, atol=1e-12)
        nosplit = helpers.orc_params_from(p)
        nosplit.splitMatrixBiggerThanThis = 1 << 62
        want1 = oracle.aligned_pairs_with_indels(om, nosplit, sx, sy, a, rl, rr)
        for key, w in zip(("bandingM", "bandingX", "bandingY"), want1):
            g = _parse_list(got[key])
            assert g.shape == w.shape and np.array_equal(g[:, 1:], w[::-1, 1:]), (i, key)
            assert g.shape[0] == 0 or np.abs(g[:, 0] - w[::-1, 0]).max() <= PINT_TOL
        assert got["banding"] == got["bandingM"]
        np.testing.assert_allclose(np.array([float.fromhex(v) for v in got["bandingE"]]), oracle.expectations(om, nosplit, sx, sy, a, rl, rr),
                                   rtol=1e-9, atol=1e-12)
    f = lines[k].split()
    assert f[0] == "total"
    np.testing.assert_allclose(np.array([float.fromhex(v) for v in f[1:]]), total, rtol=1e-9, atol=1e-12)
