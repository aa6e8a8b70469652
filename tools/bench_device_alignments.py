"""Device decoders (cpb_batch_ordered_chain, cpb_batch_mea) against libcpecan.so's host functions on the same lists, through
cpecan_b200/lib/bench_decode (tools/bench_decode.c): per workload the device decode time (median of --reps synchronised calls after a
warm-up), the host functions on --threads host threads, timed in C, the bytes a caller fetches (the posterior cloud against the alignment
list), and how many of all pairs differ.

  C2 library defaults, ALIGNED_PAIRS: reweight + chain      C2 library defaults, INDELS: MEA + left shift
  C2 cPecanRealign's parameters (trim 0, expansion 4, split 10), ALIGNED_PAIRS: chain
  C3 library defaults, ALIGNED_PAIRS: chain                 C3 library defaults, INDELS: MEA + left shift (--no-c3-mea skips it)

Writes one JSON document (with the card's name and power limit) to --out.

  python tools/bench_device_alignments.py --out profiles/r4_device_alignments.json [--scale 0.01]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import cpecan_b200 as cp  # noqa: E402
from cpecan_b200 import synth  # noqa: E402

EXE = os.path.join(ROOT, "cpecan_b200", "lib", "bench_decode")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [v.strip() for v in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:
        return {"name": "unknown (%s)" % e}


def write_seqs(path, packed):
    n = len(packed["xOff"]) - 1
    with open(path, "wb") as f:
        f.write(np.int64(n).tobytes())
        f.write(np.ascontiguousarray(packed["xOff"], dtype=np.int64).tobytes())
        f.write(np.ascontiguousarray(packed["yOff"], dtype=np.int64).tobytes())
        f.write(np.ascontiguousarray(packed["seqX"], dtype=np.uint8)[: int(packed["xOff"][-1])].tobytes())
        f.write(np.ascontiguousarray(packed["seqY"], dtype=np.uint8)[: int(packed["yOff"][-1])].tobytes())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the pair counts")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--threads", type=int, default=16)
    ap.add_argument("--no-c3-mea", action="store_true")
    ap.add_argument("--timeout", type=float, default=600, help="seconds per workload; a workload that takes longer is reported as not measured")
    args = ap.parse_args()
    p = cp.pairwiseAlignmentBandingParameters_construct()
    trim, exp, split, gap = int(p.constraintDiagonalTrim), int(p.diagonalExpansion), int(p.splitMatrixBiggerThanThis), float(p.gapGamma)
    n2, n3 = max(1, int(100000 * args.scale)), max(1, int(1250 * args.scale))
    result = {"card": card(), "host_threads": args.threads, "reps": args.reps, "workloads": []}
    with tempfile.TemporaryDirectory() as tmp:
        c2, c3 = os.path.join(tmp, "c2.bin"), os.path.join(tmp, "c3.bin")
        write_seqs(c2, synth.evolved_pairs(n2, 1000, seed=2, trim=0, expansion=0))
        write_seqs(c3, synth.evolved_pairs(n3, 100000, seed=3, trim=0, expansion=0, batch=64))
        runs = [("C2: %d x 1 kb, library defaults, ALIGNED_PAIRS: reweight + chain (matchGamma 0.85)" % n2, c2, "chain", trim, exp, split, 0.85, gap),
                ("C2: %d x 1 kb, library defaults, INDELS: MEA + left shift" % n2, c2, "mea", trim, exp, split, gap, -1),
                ("C2: %d x 1 kb, cPecanRealign's parameters, ALIGNED_PAIRS: chain (matchGamma 0.85)" % n2, c2, "chain", 0, 4, 10, 0.85, -1),
                ("C3: %d x 100 kb, library defaults, ALIGNED_PAIRS: chain (matchGamma 0.85)" % n3, c3, "chain", trim, exp, split, 0.85, -1)]
        if not args.no_c3_mea:
            runs.append(("C3: %d x 100 kb, library defaults, INDELS: MEA + left shift" % n3, c3, "mea", trim, exp, split, gap, -1))
        # cPecanRealign's narrow bands around anchors of every column put many posteriors within 2e-8 of an integer weight, which the
        # run recomputes with the host's libm: more than the default fix-up buffer holds for 100 000 pairs
        env = dict(os.environ, CPB_PINT_FIXUP_CAP=os.environ.get("CPB_PINT_FIXUP_CAP", "4000000"))
        for name, path, kind, t, e, s, gamma, rw in runs:
            cmd = [EXE, path, kind, str(t), str(e), str(s), repr(gamma), repr(rw), str(args.threads), str(args.reps)]
            print("%s ..." % name, file=sys.stderr, flush=True)
            try:
                out = subprocess.run(cmd, stdout=subprocess.PIPE, text=True, timeout=args.timeout, env=env)  # progress goes to stderr as it comes
            except subprocess.TimeoutExpired:
                entry = {"workload": name, "status": "not measured: did not finish within %d s" % args.timeout}
            else:
                if out.returncode in (0, 1) and out.stdout.strip():
                    entry = dict(workload=name, **json.loads(out.stdout.strip().splitlines()[-1]))
                else:
                    entry = {"workload": name, "error": "exit code %d" % out.returncode}
            print(json.dumps(entry), flush=True)
            result["workloads"].append(entry)
    if args.no_c3_mea:
        result["workloads"].append({"workload": "C3: %d x 100 kb, library defaults, INDELS: MEA + left shift" % n3, "status": "not measured"})
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    if any(w.get("pairs_differing") or "error" in w for w in result["workloads"]):
        sys.exit("device alignments differ from the host's, or a workload failed")


if __name__ == "__main__":
    main()
