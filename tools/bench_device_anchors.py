"""Device anchoring (cpb_batch_create_anchored) against the host anchorer of libcpecan.so, on three workloads:

  C2  100 000 x 1 kb evolved pairs, library defaults
  C3  1 250 x 100 kb evolved pairs, library defaults
  C5  the 2 016 pairs of 64 x 10 kb family members, library defaults

For each: the host's getBlastPairsForPairwiseAlignmentParameters over all pairs on every host thread (ctypes calls release the GIL),
the time of cpb_batch_create_anchored minus that of cpb_batch_create given the host's anchors (both synchronise before they return;
median of --reps alternating calls), and whether the device's anchors equal the host's (every pair is compared, not a sample).
Writes one JSON document (with the card's name and power limit) to --out.

  python tools/bench_device_anchors.py --out profiles/r3_device_anchors.json [--scale 0.01]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cpecan_b200 as cp  # noqa: E402
from cpecan_b200 import synth  # noqa: E402
from host_anchors import HostAnchorer  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [v.strip() for v in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers are still reported, marked as coming from an unidentified card
        return {"name": "unknown (%s)" % e}


def workloads(scale):
    p = cp.pairwiseAlignmentBandingParameters_construct()
    n = max(1, int(100000 * scale))
    packed = synth.evolved_pairs(n, 1000, seed=2, trim=0, expansion=0)
    yield "C2: %d x 1 kb, library defaults" % n, [synth.unpack(packed, i)[:2] for i in range(n)], p
    n = max(1, int(1250 * scale))
    packed = synth.evolved_pairs(n, 100000, seed=3, trim=0, expansion=0, batch=64)
    yield "C3: %d x 100 kb, library defaults" % n, [synth.unpack(packed, i)[:2] for i in range(n)], p
    k = max(4, int(round(64 * scale ** 0.5)))
    rng = np.random.default_rng(5)
    anc = synth.random_sequence(rng, 10000, acgt_only=True)
    members = [synth.evolve_with_alignment(rng, anc)[0].encode() for _ in range(k)]
    yield "C5: all pairs of %d x 10 kb (%d pairs)" % (k, k * (k - 1) // 2), [(members[i], members[j]) for i in range(k) for j in range(i + 1, k)], p


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the pair counts (C5: of the sequence count squared)")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    host = HostAnchorer()
    ctx = cp.Context(0)
    threads = os.cpu_count() or 1
    result = {"card": card(), "host_threads": threads, "workloads": []}
    for name, pairs, p in workloads(args.scale):
        sx, sy = [x for x, _ in pairs], [y for _, y in pairs]
        hp = host.params(p)
        with ThreadPoolExecutor(threads) as pool:
            t0 = time.perf_counter()
            handles = list(pool.map(lambda q: host.blast_pairs(q[0], q[1], hp), pairs, chunksize=64))
            host_s = time.perf_counter() - t0
        want = [host.read(h) for h in handles]
        cp.Batch.anchored(ctx, sx[:1], sy[:1], p).close()  # module load and first allocations
        dev_s, ref_s = [], []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            dev = cp.Batch.anchored(ctx, sx, sy, p)
            dev_s.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            ref = cp.Batch(ctx, sx, sy, [w if len(w) else [] for w in want])
            ref_s.append(time.perf_counter() - t0)
            ref.close()
            off, tri = dev.fetch_anchors()
            dev.close()
        differ = [i for i in range(len(pairs)) if not np.array_equal(tri[off[i]:off[i + 1]], want[i])]
        entry = {
            "workload": name,
            "pairs": len(pairs),
            "anchors": int(off[-1]),
            "host_anchoring_ms": round(1e3 * host_s, 1),
            "create_anchored_ms": round(1e3 * float(np.median(dev_s)), 1),
            "create_with_host_anchors_ms": round(1e3 * float(np.median(ref_s)), 1),
            "device_anchoring_ms": round(1e3 * (float(np.median(dev_s)) - float(np.median(ref_s))), 1),
            "pairs_checked": len(pairs),
            "pairs_differing": len(differ),
            "first_differing": differ[:10],
        }
        print(json.dumps(entry), flush=True)
        result["workloads"].append(entry)
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    if any(w["pairs_differing"] for w in result["workloads"]):
        sys.exit("device anchors differ from the host's")


if __name__ == "__main__":
    main()
