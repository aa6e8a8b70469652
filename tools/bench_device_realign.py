"""cPecanRealign with the realignment decoded on the device (this tree's cpecan_b200/lib) against a baseline build that decodes on the host
(--baseline DIR: a lib directory holding cPecanRealign, libcpecan.so and libcpecan_b200.so of the commit to compare with, built beforehand).

Every workload is run once per build to warm up, then --reps times per build, alternating.  Per build it records the process wall time
(median), the $CPECAN_HOST_TIMING stages of the median run, and the bytes copied device to host (cloud triples on the host route, cigar
operations and scores on the device route, both from the stage lines); per workload whether stdout and the posterior files are the same
bytes.  A run that fails (e.g. on the weight fix-up buffer, CPB_PINT_FIXUP_CAP) is recorded with its message.  Writes one JSON document
with the card's name and power limit to --out.

  python tools/bench_device_realign.py --baseline DIR --out profiles/r6_device_realign.json [--scale 0.01]
"""
import argparse
import hashlib
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from cpecan_b200 import synth  # noqa: E402
from bench_device_alignments import card  # noqa: E402

NEW = os.path.join(ROOT, "cpecan_b200", "lib", "cPecanRealign")


def write_inputs(fa, cig, n, length):
    """bench.py's e2e_cli recipe: evolved pairs (seed 0xC1, trim 0, expansion 4); the input alignment is the anchor columns, the equally
    long stretches between them as mismatched columns, the rest as a deletion and / or an insertion"""
    packed = synth.evolved_pairs(n, length, seed=0xC1, trim=0, expansion=4)
    with open(fa, "w") as f, open(cig, "w") as g:
        for i in range(n):
            sx, sy, a = synth.unpack(packed, i)
            f.write(">x%d\n%s\n>y%d\n%s\n" % (i, sx.decode(), i, sy.decode()))
            xs, ys = a[:, 0], a[:, 1]
            if xs.size == 0:
                continue
            gx, gy = np.diff(xs) - 1, np.diff(ys) - 1
            ops, cur = [], int(xs[0])
            for k in np.nonzero(gx != gy)[0]:
                both = int(min(gx[k], gy[k]))
                ops.append(("M", int(xs[k]) - cur + 1 + both))
                if gx[k] > both:
                    ops.append(("D", int(gx[k]) - both))
                if gy[k] > both:
                    ops.append(("I", int(gy[k]) - both))
                cur = int(xs[k + 1])
            ops.append(("M", int(xs[-1]) - cur + 1))
            g.write("cigar: y%d %d %d + x%d %d %d + 1.0%s\n" % (i, int(ys[0]), int(ys[-1]) + 1, i, int(xs[0]), int(xs[-1]) + 1,
                                                              "".join(" %s %d" % o for o in ops)))


def digest(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def run_once(exe, fa, cig, args, tmp, tag, timeout):
    """-> (wall seconds, stage ms, device-to-host bytes, {output: sha256}) or a failure message"""
    files = {opt: os.path.join(tmp, "%s%s.tsv" % (tag, opt)) for opt in ("--outputPosteriorProbs", "--outputAllPosteriorProbs") if opt in args}
    cmd = [exe]
    it = iter(args)
    for a in it:
        cmd.append(a)
        if a in files:
            next(it)
            cmd.append(files[a])
    out_path = os.path.join(tmp, tag + ".out")
    env = dict(os.environ, CPECAN_HOST_TIMING="1")
    t0 = time.perf_counter()
    try:
        with open(cig) as g, open(out_path, "w") as o:
            p = subprocess.run(cmd + [fa], stdin=g, stdout=o, stderr=subprocess.PIPE, text=True, timeout=timeout, env=env)
    except subprocess.TimeoutExpired:
        return "did not finish within %d s" % timeout
    wall = time.perf_counter() - t0
    if p.returncode != 0:
        return "exit code %d: %s" % (p.returncode, p.stderr.strip()[-400:])
    stages = {}
    for m in re.finditer(r"^\[cPecanRealign\] (.+?)\s+([0-9.]+) ms$", p.stderr, re.M):
        stages[m.group(1)] = round(stages.get(m.group(1), 0.0) + float(m.group(2)), 1)
    d2h = sum(12 * int(m.group(1)) for m in re.finditer(r"copy \+ reference order of (\d+) triples", p.stderr))
    d2h += sum(int(m.group(1)) for m in re.finditer(r"device to host: \d+ cigar operations, (\d+) bytes in all", p.stderr))
    outputs = {"stdout": digest(out_path)}
    outputs.update({opt: digest(path) for opt, path in files.items()})
    return wall, stages, d2h, outputs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline", required=True, help="lib directory of the build to compare with (its cPecanRealign)")
    ap.add_argument("--out", required=True)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the pair counts")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--timeout", type=float, default=900)
    args = ap.parse_args()
    base = os.path.join(os.path.abspath(args.baseline), "cPecanRealign")
    for exe in (NEW, base):
        if not os.path.exists(exe):
            sys.exit("%s is not built" % exe)
    sc = lambda n: max(1, int(n * args.scale))  # noqa: E731
    workloads = [
        ("e2e_cli: %d x 1 kb, the program's defaults" % sc(20000), sc(20000), 1000, []),
        ("e2e_cli with --rescoreByIdentity", sc(20000), 1000, ["--rescoreByIdentity"]),
        ("%d x 1 kb in passes of --batchBases 40000000" % sc(100000), sc(100000), 1000, ["--batchBases", "40000000"]),
        ("%d x 10 kb" % sc(2000), sc(2000), 10000, []),
        ("%d x 1 kb with both posterior files and --rescoreByPosteriorProb" % sc(2000), sc(2000), 1000,
         ["--outputPosteriorProbs", "FILE", "--outputAllPosteriorProbs", "FILE", "--rescoreByPosteriorProb"]),
    ]
    result = {"card": card(), "reps": args.reps, "baseline": "the parent commit's cPecanRealign (host decode of the fetched posteriors)",
              "device_route": "this tree's cPecanRealign (getRealignedCigarsUsingAnchorsBatch)", "workloads": []}
    with tempfile.TemporaryDirectory() as tmp:
        for name, n, length, extra in workloads:
            print("%s ..." % name, file=sys.stderr, flush=True)
            fa, cig = os.path.join(tmp, "seqs.fa"), os.path.join(tmp, "aln.cigar")
            write_inputs(fa, cig, n, length)
            entry = {"workload": name, "args": extra}
            runs = {"baseline": [], "device": []}
            failed = {}
            for rep in range(args.reps + 1):  # the first is the warm-up
                for key, exe in (("baseline", base), ("device", NEW)):
                    if key in failed:
                        continue
                    r = run_once(exe, fa, cig, extra, tmp, "%s%d" % (key, rep), args.timeout)
                    if isinstance(r, str):
                        failed[key] = r
                    elif rep > 0:
                        runs[key].append(r)
            for key in runs:
                if key in failed:
                    entry[key] = {"status": "failed: " + failed[key]}
                    continue
                med = sorted(runs[key], key=lambda r: r[0])[len(runs[key]) // 2]
                entry[key] = {"s_process_median": round(statistics.median(r[0] for r in runs[key]), 3),
                              "s_process_all": [round(r[0], 3) for r in runs[key]], "stages_ms_of_median_run": med[1],
                              "bytes_device_to_host": med[2]}
            if not failed:
                outs = [r[3] for key in runs for r in runs[key]]
                entry["outputs_identical"] = all(o == outs[0] for o in outs)
                entry["speedup_process"] = round(entry["baseline"]["s_process_median"] / entry["device"]["s_process_median"], 3)
            print(json.dumps(entry), flush=True)
            result["workloads"].append(entry)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    if any(w.get("outputs_identical") is False for w in result["workloads"]):
        sys.exit("outputs differ between the builds")


if __name__ == "__main__":
    main()
