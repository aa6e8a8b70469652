"""Cigars in on the flat C-ABI: device against host route, through cpecan_b200/lib/bench_cigar_inputs (tools/bench_cigar_inputs.c).

Two comparisons on every workload, with cPecanRealign's parameters (trim 0, expansion 4, split 10) and the five-state default model:
- anchors: convertPairwiseForwardStrandAlignmentToAnchorPairs + columns_match on --threads host threads, then cpb_batch_create, against
  cpb_batch_create_from_cigars;
- rescoring (cPecanRealign --rescoreOriginalAlignment --rescoreByPosteriorProb): list 0 fetched in reference order, then weighing, score and
  cigar on --threads host threads, against cpb_batch_alignments_from_cigars, the score and the cigar build on the device.  The ALIGNED_PAIRS
  run both start from is timed on its own.
Workloads: 20 000 x 1 kb (the e2e_cli shape), 2 000 x 10 kb, and 100 000 x 1 kb in five batches of 20 000.  Times are the median, min and
max of --reps repetitions after a warm-up; every pair's anchors, score bits and cigar are compared between the routes, and the bytes each
route moves across the link are counted.  A workload that fails or does not finish within --timeout is reported as not measured, with the
reason.  Writes one JSON document (with the card's name and power limit) to --out.

  python tools/bench_cigar_inputs.py --out profiles/r7_cigar_inputs.json [--scale 0.01]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_device_alignments import card  # noqa: E402

EXE = os.path.join(ROOT, "cpecan_b200", "lib", "bench_cigar_inputs")
WORKLOADS = [("e2e_cli: 20 000 x 1 kb", 20000, 1000, 20000), ("2 000 x 10 kb", 2000, 10000, 2000),
             ("100 000 x 1 kb in five batches of 20 000", 100000, 1000, 20000)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the pair counts")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--threads", type=int, default=16)
    ap.add_argument("--timeout", type=float, default=900, help="seconds; a workload that takes longer is reported as not measured")
    args = ap.parse_args()
    result = {"card": card(), "host_threads": args.threads, "reps": args.reps, "workloads": []}
    for name, n, length, batch in WORKLOADS:
        n, batch = max(1, int(n * args.scale)), max(1, int(batch * args.scale))
        cmd = [EXE, str(n), str(length), str(batch), str(args.threads), str(args.reps)]
        print("%s ..." % name, file=sys.stderr, flush=True)
        try:
            out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=args.timeout)
        except subprocess.TimeoutExpired:
            entry = {"workload": name, "status": "not measured: did not finish within %d s" % args.timeout}
        else:
            sys.stderr.write(out.stderr)
            if out.returncode in (0, 1) and out.stdout.strip():
                entry = dict(workload=name, **json.loads(out.stdout.strip().splitlines()[-1]))
            else:
                entry = {"workload": name, "status": "not measured: exit code %d: %s" % (out.returncode, out.stderr.strip()[-400:])}
        print(json.dumps(entry), flush=True)
        result["workloads"].append(entry)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    if any(w.get("pairs_differing") for w in result["workloads"]):
        sys.exit("the device route differs from the host route")


if __name__ == "__main__":
    main()
