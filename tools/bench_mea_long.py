"""The MEA with left shift on C2 (100 000 x 1 kb) and C3 (1 250 x 100 kb), library defaults, INDELS, through cpecan_b200/lib/bench_decode
(tools/bench_decode.c):

  * this build: device decode (median of three synchronised cpb_batch_mea calls after a warm-up), the host functions
    (getMaximalExpectedAccuracyPairwiseAlignment + leftShiftAlignment) on --threads host threads over the lists in the reference's order,
    and every pair compared (triples and the bits of alignmentScore);
  * device decode of this build and of --baseline DIR (a lib directory holding libcpecan_b200.so of the commit to compare with, built
    beforehand), device only, alternating process by process, --rounds times each; a baseline run that takes longer than --timeout is
    recorded as not finished and not repeated.

Writes one JSON document with the card's name and power limit (read in the same call) to --out.

  python tools/bench_mea_long.py --baseline DIR --out profiles/r8_mea_long.json [--scale 0.01]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import cpecan_b200 as cp  # noqa: E402
from cpecan_b200 import synth  # noqa: E402
from bench_device_alignments import EXE, card, write_seqs  # noqa: E402


def run(cmd, env, timeout):
    try:
        out = subprocess.run(cmd, stdout=subprocess.PIPE, text=True, timeout=timeout, env=env)
    except subprocess.TimeoutExpired:
        return {"status": "not measured: did not finish within %d s" % timeout}
    if out.returncode in (0, 1) and out.stdout.strip():
        return json.loads(out.stdout.strip().splitlines()[-1])
    return {"error": "exit code %d" % out.returncode}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline", required=True, help="lib directory of the build to compare with")
    ap.add_argument("--out", required=True)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the pair counts")
    ap.add_argument("--threads", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--timeout", type=float, default=600, help="seconds per process")
    args = ap.parse_args()
    baseline = os.path.abspath(args.baseline)
    if not os.path.exists(os.path.join(baseline, "libcpecan_b200.so")):
        sys.exit("no libcpecan_b200.so under %s" % baseline)
    p = cp.pairwiseAlignmentBandingParameters_construct()
    trim, exp, split, gap = int(p.constraintDiagonalTrim), int(p.diagonalExpansion), int(p.splitMatrixBiggerThanThis), float(p.gapGamma)
    n2, n3 = max(1, int(100000 * args.scale)), max(1, int(1250 * args.scale))
    result = {"card": card(), "host_threads": args.threads, "rounds": args.rounds, "baseline": "parent commit's libcpecan_b200.so",
              "device_ms": "median of three synchronised cpb_batch_mea calls (MEA + left shift) after a warm-up, per process", "workloads": []}
    this_env = dict(os.environ)
    base_env = dict(os.environ, LD_LIBRARY_PATH=baseline + os.pathsep + os.environ.get("LD_LIBRARY_PATH", ""))
    with tempfile.TemporaryDirectory() as tmp:
        c2, c3 = os.path.join(tmp, "c2.bin"), os.path.join(tmp, "c3.bin")
        write_seqs(c2, synth.evolved_pairs(n2, 1000, seed=2, trim=0, expansion=0))
        write_seqs(c3, synth.evolved_pairs(n3, 100000, seed=3, trim=0, expansion=0, batch=64))
        for name, path in (("C2: %d x 1 kb, library defaults, INDELS: MEA + left shift" % n2, c2),
                           ("C3: %d x 100 kb, library defaults, INDELS: MEA + left shift" % n3, c3)):
            cmd = lambda threads, reps: [EXE, path, "mea", str(trim), str(exp), str(split), repr(gap), "-1", str(threads), str(reps)]  # noqa: E731
            print("%s: this build with the host arm ..." % name, file=sys.stderr, flush=True)
            entry = {"workload": name, "this_build": run(cmd(args.threads, 3), this_env, args.timeout)}
            mine, base = [], []
            for r in range(args.rounds):
                print("%s: device only, round %d ..." % (name, r + 1), file=sys.stderr, flush=True)
                mine.append(run(cmd(0, 3), this_env, args.timeout))
                if not base or "device_ms" in base[-1]:
                    base.append(run(cmd(0, 3), base_env, args.timeout))
            entry["device_only"] = {"this_build_ms": [m.get("device_ms", m.get("status", m.get("error"))) for m in mine],
                                    "baseline_ms": [b.get("device_ms", b.get("status", b.get("error"))) for b in base]}
            for key, runs in (("this_build_median_ms", mine), ("baseline_median_ms", base)):
                ms = [m["device_ms"] for m in runs if "device_ms" in m]
                entry["device_only"][key] = statistics.median(ms) if len(ms) == len(runs) and ms else None
            print(json.dumps(entry), flush=True)
            result["workloads"].append(entry)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    if any(w["this_build"].get("pairs_differing") or "pairs_checked" not in w["this_build"] for w in result["workloads"]):
        sys.exit("device alignments differ from the host's, or this build did not finish a workload")


if __name__ == "__main__":
    main()
