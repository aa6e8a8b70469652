#!/usr/bin/env python
"""bench.py -- headline measurement of the cPecan pair-HMM hot path on B200.

Metric (BASELINE.json): GCUPS (band cells per second / 1e9, each cell counted once, SURVEY.md section 8d) and
pairs/s of banded forward-backward + posterior on `configs[1]`: 100 000 synthetic 1 kb evolved pairs,
StateMachine5, library-default band and posterior threshold 0.01.  One "step" = one pass of the whole hot path
(band builder -> forward -> backward -> totals -> posterior scan/compaction) over the batch.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--pairs P] [--impl reference] [--dump-outputs DIR]

value : inputs resident in HBM, CUDA-event time on the launching stream over K steps, max over ranks.
e2e   : the same pass through the C-ABI with HOST buffers (pinned): cpb_batch_create (H2D) + cpb_batch_run +
        cpb_batch_fetch_pairs (D2H) inside the timed region, K steps.
--dump-outputs DIR : after the timed steps, what the last one computed goes to DIR/*.npy (dump_outputs), so that two builds
        can be compared output for output on the same seeded inputs.
--impl reference : the reference's own CPU implementation (oracle/_ref when it was built, else the plain-C port)
        on all host cores over a bounded sample of the same workload.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "GCUPS (banded fwd-bwd+posterior)"
UNIT = "GCUPS"
WORKLOAD = "100k x 1 kb evolved pairs (randomSequences-style, ~10% divergence), StateMachine5, lib-default band (expansion 20, trim 14), threshold 0.01"
# DESIGN.md section 5, per band cell (five states, aligned-pairs mode).  One sweep = 13 transition adds + 8 logAdds of 8 separately
# rounded FP64 operations (1 subtract, 3 multiplies, 4 adds; contraction to FMA is not allowed) = 77; the backward sweep adds the
# F + B sum = 78; forward + backward = 155 (SURVEY.md section 8d's 280 "FLOP" counted compares and selects, which are not FP64 work).
OPS_FORWARD, OPS_BACKWARD = 77.0, 78.0
# HBM: what the two sweeps have to move per cell -- forward writes F.M (8 B) + 1/10 of the full cell (4 B); backward reads F.M (8 B)
# and 1/10 of the full cell (4 B) and writes F + B (8 B); (the posterior scan reads those 8 B again in its own kernel)
ALG_BYTES_FORWARD, ALG_BYTES_BACKWARD = 12.0, 20.0
# measured dram__bytes_read.sum + dram__bytes_write.sum per cell of one launch (ncu --set full, profiles/): forward, backward
DRAM_BYTES_FORWARD, DRAM_BYTES_BACKWARD = 18.8, 34.7
FP64_LANES_PER_SM = 64      # B200: 64 FP64 lanes per SM and clock; tools/ubench.cu measures 59.4 sustained (profiles/r1_ubench.txt)


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            pk = json.load(f)
        return float(pk.get("hbm_gbs", 6650.0)), float(pk.get("sm_max_mhz", 1965.0)), "measured"
    return 6650.0, 1965.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows = []
        self.index = index
        self.proc = None
        self.thread = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_inputs(n_pairs, rank, params):
    from cpecan_b200 import synth

    return synth.evolved_pairs(n_pairs, 1000, seed=0xC0FFEE + 7919 * rank, trim=int(params.constraintDiagonalTrim),
                               expansion=int(params.diagonalExpansion))


def dump_outputs(batch, out_dir, n_sample=1024):
    """The aligned pairs of the batch's last run, as cpb_batch_fetch_pairs hands them to a caller, in float64 (exact for these
    integers).  All of them would be ~1.3 GB at 100 000 pairs, so: offsets.npy, where each pair's triples start (n + 1);
    pint_sum.npy, the sum of pInt over each pair's triples (n); triples_sample.npy, the triples of a fixed, seeded sample of
    n_sample pairs in the order they are returned, columns (pair, pInt, x, y) -- about 36 MB at 1 kb pairs."""
    off, tri = batch.fetch_pairs(0)
    n = len(off) - 1
    csum = np.concatenate([[0], np.cumsum(tri[:, 0], dtype=np.int64)])
    pick = np.sort(np.random.default_rng(0).choice(n, size=min(n, n_sample), replace=False))
    sample = [np.column_stack([np.full(off[p + 1] - off[p], p), tri[off[p]:off[p + 1]]]) for p in pick]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "offsets.npy"), off.astype(np.float64))
    np.save(os.path.join(out_dir, "pint_sum.npy"), (csum[off[1:]] - csum[off[:-1]]).astype(np.float64))
    np.save(os.path.join(out_dir, "triples_sample.npy"), np.concatenate(sample or [np.zeros((0, 4))]).astype(np.float64))


def cpu_arm(packed, n_sample, threads):
    """Times the CPU implementation (reference build if present) on the first n_sample pairs of the workload.  Nothing here touches
    the product library: parameters and model come from the oracle itself, the generator is plain numpy."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    from cpecan_b200 import synth

    orc = helpers.best_oracle()
    sub = synth.subset(packed, range(n_sample))
    p = orc.default_params()
    m = helpers.ModelSpec(0).orc()  # fiveState, the reference's default model
    t0 = time.perf_counter()
    counts, _, _ = orc.batch(m, p, sub, mode=0, threads=threads)
    dt = time.perf_counter() - t0
    return orc.identity, dt, int(counts.sum())


def count_cells(packed, n_sample):
    """band cells of the first n_sample pairs, from the product's own band builder statistics (b200 arm only)"""
    import cpecan_b200 as cp
    from cpecan_b200 import synth

    ctx = cp.Context(int(os.environ.get("LOCAL_RANK", "0")))
    b = cp.Batch(ctx, None, None, packed=synth.subset(packed, range(n_sample)))
    b.run(cp.stateMachine5_construct(), cp.pairwiseAlignmentBandingParameters_construct(), cp.MODE_FORWARD)
    cells = b.stats().cells
    b.close()
    ctx.close()
    return int(cells)


def capi_arm(cp, device, stream, model, params, packed, n, barrier):
    """The same pass through the reference-named batch call of libcpecan.so (tools/bench_capi.c): strings and stLists of anchor tuples
    in, stLists of (pInt, x, y) tuples out, walked once and destructed -- beside the flat C-ABI on the same subset of the workload.
    A subset (default 20 000 pairs) because the reference's interface needs ~100 bytes of host heap per aligned pair."""
    from cpecan_b200 import synth

    exe = os.path.join(ROOT, "cpecan_b200", "lib", "bench_capi")
    if not os.path.exists(exe):
        return {"value": None, "note": "cpecan_b200/lib/bench_capi is not built"}
    sub = synth.subset(packed, range(n))
    path = "/tmp/cpecan_capi_workload_%d.bin" % os.getpid()
    with open(path, "wb") as f:
        np.asarray([n], dtype=np.int64).tofile(f)
        for k in ("xOff", "yOff", "aOff"):
            np.ascontiguousarray(sub[k], dtype=np.int64).tofile(f)
        np.ascontiguousarray(sub["seqX"][: int(sub["xOff"][-1])], dtype=np.uint8).tofile(f)
        np.ascontiguousarray(sub["seqY"][: int(sub["yOff"][-1])], dtype=np.uint8).tofile(f)
        np.ascontiguousarray(sub["anchors"][: 3 * int(sub["aOff"][-1])], dtype=np.int64).tofile(f)
    try:
        out = subprocess.run([exe, path, "2", "1"], capture_output=True, text=True, timeout=600)
        j = json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as ex:
        return {"value": None, "note": "bench_capi failed: %s" % ex}
    finally:
        os.remove(path)
    # the flat C-ABI on the same subset, for the ratio (a fresh context: same conditions as the subprocess had)
    import torch

    ctx = cp.Context(device, stream=stream.cuda_stream)
    b = cp.Batch(ctx, None, None, packed=sub)
    b.run(model, params, cp.MODE_ALIGNED_PAIRS)
    cells, n_tri = int(b.stats().cells), int(b.stats().outputTriples)
    b.close()
    out_pinned = torch.empty((max(n_tri, 1) + 1024, 3), dtype=torch.int32).pin_memory()
    barrier()
    t0 = time.perf_counter()
    for _ in range(2):
        b = cp.Batch(ctx, None, None, packed=sub)
        b.run(model, params, cp.MODE_ALIGNED_PAIRS)
        b.fetch_pairs(0, out=out_pinned.numpy())
        b.close()
    flat = (time.perf_counter() - t0) / 2
    ctx.close()
    # value: the call plus giving the lists back (what the library costs its caller); the caller's own walk over the tuples is beside it
    s_lib = j["s_call"] + j["s_destruct"]
    return {"value": cells / s_lib / 1e9, "unit": UNIT, "pairs": n, "pairs_per_s": n / s_lib, "tuples": j["tuples"],
            "s_call": j["s_call"], "s_destruct": j["s_destruct"], "s_callers_walk_over_the_tuples": j["s_walk"],
            "flat_abi_same_pairs": {"value": cells / flat / 1e9, "unit": UNIT, "s": flat},
            "ratio_capi_over_flat_time": s_lib / flat, "ratio_call_only_over_flat_time": j["s_call"] / flat,
            "api": "getAlignedPairsUsingAnchorsBatch (include/cpecan/pairwiseAligner.h), stList / stIntTuple in and out"}


def cli_arm(n, length=1000):
    """cPecanRealign itself, the program of the reference that north_star names: FASTA and cigars in, realigned cigars out, with its
    own defaults (band of +-4 around the input alignment's matching columns, split at gaps of more than 10 cells).  The input
    alignments are the anchor columns of synthetic evolved pairs; the process is started twice and the second run is timed, start to
    exit -- CUDA context creation, parsing, one device pass per --batchBases, maximal-expected-accuracy alignment, output."""
    from cpecan_b200 import synth

    exe = os.path.join(ROOT, "cpecan_b200", "lib", "cPecanRealign")
    if not os.path.exists(exe):
        return {"value": None, "note": "cpecan_b200/lib/cPecanRealign is not built"}
    packed = synth.evolved_pairs(n, length, seed=0xC1, trim=0, expansion=4)
    fa, cig = "/tmp/cpecan_cli_%d.fa" % os.getpid(), "/tmp/cpecan_cli_%d.cigar" % os.getpid()
    try:
        with open(fa, "w") as f, open(cig, "w") as g:
            for i in range(n):
                sx, sy, a = synth.unpack(packed, i)
                f.write(">x%d\n%s\n>y%d\n%s\n" % (i, sx.decode(), i, sy.decode()))
                xs, ys = a[:, 0], a[:, 1]
                if xs.size == 0:
                    continue
                # the input alignment: the anchor columns, the equally long stretches between them as mismatched columns of the same
                # match operation (what an aligner emits for substitutions), the rest as a deletion and / or an insertion
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
        wall, lines = None, 0
        for _ in range(2):
            t0 = time.perf_counter()
            with open(cig) as g:
                out = subprocess.run([exe, fa], stdin=g, capture_output=True, text=True, timeout=900)
            wall = time.perf_counter() - t0
            if out.returncode != 0:
                return {"value": None, "note": "cPecanRealign failed: %s" % out.stderr.strip()[-300:]}
            lines = sum(1 for l in out.stdout.splitlines() if l.startswith("cigar:"))
        return {"value": n / wall, "unit": "pairs/s", "pairs": n, "cigars_out": lines, "s_process": wall,
                "program": "cPecanRealign seqs.fa < alignments.cigar (its own defaults), whole process incl. CUDA context creation"}
    except Exception as ex:
        return {"value": None, "note": "cPecanRealign arm failed: %s" % ex}
    finally:
        for path in (fa, cig):
            if os.path.exists(path):
                os.remove(path)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=100000, help="pairs per GPU (weak scaling)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU work of the cpu_baseline sample")
    ap.add_argument("--capi-pairs", type=int, default=20000, help="pairs of the workload sent through the reference-named C API (e2e_capi)")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only: no end-to-end arm")
    ap.add_argument("--skip-cpu", action="store_true", help="profiling runs only: no CPU baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the aligned pairs of the last timed step to DIR/*.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the CUDA path computed: not with --impl reference")

    # Every timed pass plans its run anew (regions, bands, traceback schedule, chunks, work lists), as the first call on a new batch
    # does: the engine would otherwise keep the plan of a batch that is run again with the same parameters (what EM iterations do).
    os.environ["CPB_NO_PLAN_CACHE"] = "1"
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    threads = os.cpu_count() or 1

    if args.impl == "reference":
        # the reference's CPU path on all host cores; rank 0 only.  This arm never loads the product's libraries: parameters come from
        # the oracle, band cells are counted with the oracle's band builder.
        if rank != 0:
            return
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import helpers

        params = helpers.best_oracle().default_params()
        n_sample = max(32 * threads, 256)  # enough pairs per thread for an even load
        packed = make_inputs(n_sample, 0, params)
        ident, dt_probe, _ = cpu_arm(packed, min(8, n_sample), 1)
        per_pair = dt_probe / min(8, n_sample)
        # size each step to ~ cpu-seconds/ (steps+warmup) of wall time on all threads
        steps_total = max(args.steps + args.warmup, 1)
        budget = max(args.cpu_seconds * 4 / steps_total, 2.0)
        n_step = int(min(n_sample, max(threads, budget * threads / max(per_pair, 1e-6))))
        cells = _cells_by_oracle(packed, n_step, int(params.diagonalExpansion))
        times = []
        for i in range(args.warmup + args.steps):
            _, dt, _ = cpu_arm(packed, n_step, threads)
            if i >= args.warmup:
                times.append(dt)
        tsum = sum(times)
        assert not any("libcpecan" in line and "oracle" not in line for line in open("/proc/self/maps")), "the reference arm mapped a product library"
        gcups = cells * len(times) / tsum / 1e9
        line = {
            "impl": "reference", "metric": METRIC, "value": gcups, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tsum / len(times), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample_pairs_per_step": n_step, "host_threads": threads},
            "pairs_per_s": n_step * len(times) / tsum,
            "cpu_baseline": {"value": gcups, "unit": UNIT, "cores": threads, "kind": ident,
                             "sample": "%d pairs of the workload per step, all %d host threads" % (n_step, threads)},
            "e2e": {"value": gcups, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
        return

    import torch

    import cpecan_b200 as cp

    params = cp.pairwiseAlignmentBandingParameters_construct()
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    stream = torch.cuda.current_stream()
    ctx = cp.Context(local_rank, stream=stream.cuda_stream)
    model = cp.stateMachine5_construct(cp.fiveState)

    t_gen = time.perf_counter()
    packed = make_inputs(args.pairs, rank, params)
    t_gen = time.perf_counter() - t_gen

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm ----
    batch = cp.Batch(ctx, None, None, packed=packed)
    for _ in range(args.warmup):
        batch.run(model, params, cp.MODE_ALIGNED_PAIRS)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    phase = {"band": 0.0, "forward": 0.0, "backward": 0.0, "totals": 0.0, "posterior": 0.0}
    launches = 0
    for _ in range(args.steps):
        batch.run(model, params, cp.MODE_ALIGNED_PAIRS)
        st = batch.stats()
        phase["band"] += st.msBand
        phase["forward"] += st.msForward
        phase["backward"] += st.msBackward
        phase["totals"] += st.msTotals
        phase["posterior"] += st.msPosterior
        launches += st.kernelLaunches
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    st = batch.stats()
    cells, n_triples = int(st.cells), int(st.outputTriples)
    if args.dump_outputs and rank == 0:
        dump_outputs(batch, args.dump_outputs)
    t = torch.tensor([ms, float(cells), float(args.pairs)], dtype=torch.float64, device="cuda")
    if dist is not None:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms_all, cells_all, pairs_all = float(tmax[0]), float(tsum[1]), float(tsum[2])
    else:
        ms_all, cells_all, pairs_all = ms, float(cells), float(args.pairs)
    value = cells_all * args.steps / (ms_all * 1e-3) / 1e9
    pairs_per_s = pairs_all * args.steps / (ms_all * 1e-3)

    # ---- end-to-end arm through the C-ABI with pinned host buffers ----
    pinned = {}
    for k in ("seqX", "xOff", "seqY", "yOff", "anchors", "aOff"):
        tt = torch.from_numpy(packed[k]).pin_memory()
        pinned[k] = tt.numpy()
        pinned["_t_" + k] = tt
    out_pinned = torch.empty((max(n_triples, 1) + 1024, 3), dtype=torch.int32).pin_memory()
    h2d = int(packed["xOff"][-1] + packed["yOff"][-1] + 12 * packed["aOff"][-1])
    d2h = int(n_triples * 12)
    e2e_steps = args.steps

    def one_e2e():
        b = cp.Batch(ctx, None, None, packed=pinned)
        b.set_result_sink(0, out_pinned.numpy())  # every chunk's triples leave for the host while the next chunk computes
        b.run(model, params, cp.MODE_ALIGNED_PAIRS)
        off, tri = b.fetch_pairs(0, out=out_pinned.numpy())
        b.close()
        return int(off[-1])

    batch.close()
    wall = float("nan")
    if not args.skip_e2e:
        one_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            got = one_e2e()
        barrier()
        wall = time.perf_counter() - t0
        assert got == n_triples, "e2e arm produced %d triples, resident arm %d" % (got, n_triples)
    tw = torch.tensor([wall], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tw, op=dist.ReduceOp.MAX)
    e2e_value = cells_all * e2e_steps / float(tw[0]) / 1e9

    e2e_capi = e2e_cli = None
    if rank == 0 and world == 1 and not args.skip_e2e:
        ctx.close()  # the C API arm runs in its own process: give it the whole GPU (this context holds 70 % of HBM as scratch)
        e2e_capi = capi_arm(cp, local_rank, stream, model, params, packed, min(args.pairs, args.capi_pairs), barrier)
        e2e_cli = cli_arm(min(args.pairs, args.capi_pairs))
    if rank == 0:
        hbm_peak, sm_max, peak_src = read_peaks()
        # The dominant kernel is the backward wavefront (one launch per chunk), then the forward one.  Both are bound by the FP64 pipe --
        # a recurrence of separately rounded adds and multiplies (SURVEY.md section 8d: "compute, not tensor cores, not HBM") -- so the
        # top-level roofline is that pipe; HBM is the secondary entry, from MEASURED dram bytes per launch.
        n_launch = max(int(st.nChunks), 1)
        fwd_ms, bwd_ms = phase["forward"] / args.steps, phase["backward"] / args.steps
        fp64_peak = 148 * FP64_LANES_PER_SM * sm_max * 1e6 / 1e12  # TFLOP/s of non-fused FP64 operations at the measured maximum clock
        def leg(ms, ops, alg_bytes, dram_bytes):
            return {"ms_per_launch": ms / n_launch, "achieved": cells * ops / (ms * 1e-3) / 1e12, "frac": cells * ops / (ms * 1e-3) / 1e12 / fp64_peak,
                    "ops_per_cell": ops,
                    "hbm": {"achieved": cells * alg_bytes / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                            "frac": cells * alg_bytes / (ms * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes_per_cell": alg_bytes,
                            "measured_dram_bytes_per_cell": dram_bytes, "traffic_over_algorithmic": dram_bytes / alg_bytes}}
        bwd, fwd = leg(bwd_ms, OPS_BACKWARD, ALG_BYTES_BACKWARD, DRAM_BYTES_BACKWARD), leg(fwd_ms, OPS_FORWARD, ALG_BYTES_FORWARD, DRAM_BYTES_FORWARD)
        both_tf = cells * (OPS_FORWARD + OPS_BACKWARD) / ((fwd_ms + bwd_ms) * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_all / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "pairs_per_gpu": args.pairs, "cells_per_gpu": cells, "l2": "working set >> L2 (GBs of DP state per step)",
                       "chunks": int(st.nChunks), "blocks": int(st.nBlocks), "max_band_width": int(st.maxWidth), "datagen_s": round(t_gen, 1)},
            "pairs_per_s": pairs_per_s,
            "gpu_launches": int(launches),
            "phase_ms_per_step": {k: v / args.steps for k, v in phase.items()},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "pairs_per_s": pairs_all * e2e_steps / float(tw[0])},
            "roofline": {"bound": "fp64", "kernel": "k_backward_strip<5,1,true,4,6>", "achieved": bwd["achieved"], "peak": fp64_peak, "unit": "TFLOP/s",
                         "frac": bwd["frac"],
                         "traffic": DRAM_BYTES_BACKWARD * cells / n_launch,
                         "note": "non-fused FP64 operations (the reference's arithmetic forbids FMA contraction); peak = 148 SMs x 64 FP64 lanes x "
                                 "sm_max_mhz of MEASURED_PEAKS.json; traffic = ncu dram__bytes_read+write of one launch (bytes per cell x cells per launch)",
                         "peak_source": peak_src, "launches_per_step": n_launch,
                         # what this instruction mix reaches with the band logic taken away (tools/ubench_step.cu on one B200, committed in
                         # profiles/r2_variants.txt): the forward step alone, every lane busy on every step
                         "bare_step_ceiling": {"forward_g_cells_per_s": 96.0, "at": "4 CTAs/SM, 110 registers", "saturates_at": 108.0,
                                               "source": "profiles/r2_variants.txt (tools/ubench_step.cu), a measurement of round 2, not of this run"},
                         "k_backward_strip": bwd, "k_forward_strip": fwd,
                         "forward_plus_backward": {"achieved": both_tf, "frac": both_tf / fp64_peak, "ops_per_cell": OPS_FORWARD + OPS_BACKWARD,
                                                   # round 1 counted 170 FP64 instructions per cell (with the directed-rounding add of the
                                                   # segment lookup): the same time on that count, for comparison with its 0.26
                                                   "frac_counting_170": both_tf / fp64_peak * 170.0 / (OPS_FORWARD + OPS_BACKWARD)}},
        }
        if e2e_capi is not None:
            line["e2e_capi"] = e2e_capi
        if e2e_cli is not None:
            line["e2e_cli"] = e2e_cli
        # CPU baseline on a bounded sample of the same workload
        try:
            if args.skip_cpu:
                raise RuntimeError("skipped (--skip-cpu)")
            n_probe = 8
            ident, dt_probe, _ = cpu_arm(packed, n_probe, 1)
            per_pair = dt_probe / n_probe
            n_sample = int(min(args.pairs, max(threads, args.cpu_seconds * threads / max(per_pair, 1e-6))))
            ident, dt, _ = cpu_arm(packed, n_sample, threads)
            sample_cells = count_cells(packed, n_sample)
            line["cpu_baseline"] = {"value": sample_cells / dt / 1e9, "unit": UNIT, "cores": threads, "kind": ident,
                                    "sample": "first %d pairs of the workload, %d host threads, %.1f s" % (n_sample, threads, dt),
                                    "single_core_gcups": count_cells(packed, n_probe) / dt_probe / 1e9}
        except Exception as ex:  # the baseline is reported, never required for the GPU number
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": threads, "kind": "unavailable", "sample": str(ex)}
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def _has_gpu():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


def _cells_by_oracle(packed, n, expansion):
    """band cells of the first n pairs from the oracle's band builder (band_construct, impl/pairwiseAligner.c:183-234)"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    from cpecan_b200 import synth

    orc = helpers.best_oracle()
    total = 0
    for i in range(n):
        sx, sy, a = synth.unpack(packed, i)
        b = orc.band(a, len(sx), len(sy), expansion)
        total += int(((b[:, 2] - b[:, 1]) // 2 + 1).sum())
    return total


if __name__ == "__main__":
    main()
