"""cPecanEm --updateTheBand on the device against the host route, through cpecan_b200/lib/bench_band_update (tools/bench_band_update.c).

Workload C4: 50 000 x 2 kb evolved pairs, five-state default model, cPecanEm's band (trim 0, expansion 10, split 3000^2).  Reports the EM
iteration time with and without the update, the update's parts (ALIGNED_PAIRS run, reweight, chain, anchor conversion with its
device-to-host copy), the host route for the same update (reference-order lists fetched, reweightAlignedPairs2 + filterPairwiseAlignment-
ToMakePairsOrdered + cigar anchors on --threads host threads, a new batch created), the bytes each route moves across the link, and the
number of pairs whose device anchors differ from the host route's.  A workload that fails or does not finish within --timeout is reported
as not measured, with the reason.  Writes one JSON document (with the card's name and power limit) to --out.

  python tools/bench_band_update.py --out profiles/r5_band_update.json [--scale 0.01]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from cpecan_b200 import synth  # noqa: E402
from bench_device_alignments import card, write_seqs  # noqa: E402

EXE = os.path.join(ROOT, "cpecan_b200", "lib", "bench_band_update")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the pair count")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--threads", type=int, default=16)
    ap.add_argument("--trim", type=int, default=0)
    ap.add_argument("--timeout", type=float, default=900, help="seconds; a workload that takes longer is reported as not measured")
    args = ap.parse_args()
    n = max(1, int(50000 * args.scale))
    result = {"card": card(), "host_threads": args.threads, "reps": args.reps, "workloads": []}
    name = "C4: %d x 2 kb, five-state default model, cPecanEm's band (trim %d, expansion 10, split 3000^2)" % (n, args.trim)
    # narrow bands around anchors of every column put many posteriors within 2e-8 of an integer weight, which the run recomputes with the
    # host's libm: more than the default fix-up buffer holds at this size
    env = dict(os.environ, CPB_PINT_FIXUP_CAP=os.environ.get("CPB_PINT_FIXUP_CAP", "4000000"))
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "c4.bin")
        write_seqs(path, synth.evolved_pairs(n, 2000, seed=4, trim=0, expansion=0))
        cmd = [EXE, path, str(args.trim), str(args.threads), str(args.reps)]
        print("%s ..." % name, file=sys.stderr, flush=True)
        try:
            out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=args.timeout, env=env)
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
        sys.exit("device anchors differ from the host route's")


if __name__ == "__main__":
    main()
