"""Align and predict from Python lists: the two-step route (`alignment.nw_align` -> `insert_gaps` -> `Predictor.submit_structures`)
against the fused route (`Predictor.submit_pairs`, the traceback writes the contact-map query frame), on configs[4]-distribution
chunks of 16,384 (query, target, coordinates) pairs, alternated in one process.  Reports end-to-end proteins/s of both routes, the
host time of each Python step of the two-step route (including the `AlignmentResult` objects `align_pairs` builds), the kernel time
of the alignment stage from the stage profile, and the largest score difference between the routes.  The card's name and power
limit are read in the same call.

  python tools/pairs_bench.py [--pairs 16384] [--chunks 3] [--reps 3] [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mdf_pkg  # noqa: E402

mdf_pkg.load()
from metagenomic_deepfri_b200 import alignment, predict, synth  # noqa: E402

B62 = (alignment.BLOSUM62_ALPHABET, alignment.BLOSUM62)
THR, GEN = 10.0, 2


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return "nvidia-smi unavailable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=16384)
    ap.add_argument("--chunks", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    procs = min(16, os.cpu_count() or 1)
    chunks = []
    for k in range(args.chunks):
        wl = synth.keyed_workload_parallel(np.arange(k * args.pairs, (k + 1) * args.pairs), 5, procs)
        chunks.append((list(wl.query_seqs), [t.replace("-", "") for t in wl.gapped_target], list(wl.coords)))
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "mf.onnx")
        synth.write_gcn_model(path, synth.GCNConfig())
        pred = predict.Predictor(path)
        host = {"nw_align": [], "insert_gaps": [], "AlignmentResult": [], "submit_structures+wait": []}

        def two_step(c):
            qs, ts, cs = c
            t0 = time.perf_counter()
            _, ops = alignment.nw_align(qs, ts, scoring_matrix=B62)
            t1 = time.perf_counter()
            gapped = [alignment.insert_gaps(q, t, o) for q, t, o in zip(qs, ts, ops)]
            t2 = time.perf_counter()
            y = pred.submit_structures(qs, [g[0] for g in gapped], [g[1] for g in gapped], cs, THR, GEN).wait()
            t3 = time.perf_counter()
            # what align_pairs builds per pair on top (identity + AlignmentResult, which runs insert_gaps once more): timed, not
            # part of the two-step route's end-to-end time
            [alignment.AlignmentResult(f"q{i}", q, f"t{i}", t, o, alignment._stats(o, q, t)[0], 1.0, 1.0)
             for i, (q, t, o) in enumerate(zip(qs, ts, ops))]
            t4 = time.perf_counter()
            for k, dt in zip(host, (t1 - t0, t2 - t1, t4 - t3, t3 - t2)):
                host[k].append(dt * 1e3)
            return y, t3 - t0

        def fused(c):
            qs, ts, cs = c
            t0 = time.perf_counter()
            y = pred.submit_pairs(qs, ts, cs, B62, threshold=THR, generated_contacts=GEN).wait()[0]
            return y, time.perf_counter() - t0

        for c in chunks:                                    # warm-up: every chunk through both routes
            two_step(c)
            fused(c)
        for k in host:
            host[k].clear()
        times = {"two_step": [], "fused": []}
        worst = 0.0
        for _ in range(args.reps):
            for c in chunks:
                ya, ta = two_step(c)
                yb, tb = fused(c)
                times["two_step"].append(ta)
                times["fused"].append(tb)
                worst = max(worst, float(np.abs(ya - yb).max()))
        ctx = pred._ctx
        ctx.profile(True)
        pred.submit_pairs(*chunks[0], B62, threshold=THR, generated_contacts=GEN).wait()
        stages = ctx.profile_report()
        ctx.profile(False)
        pred.close()
    cells = float(sum(len(q) * len(t) for q, t in zip(chunks[0][0], chunks[0][1])))
    res = {
        "card": card(),
        "pairs_per_chunk": args.pairs, "chunks": args.chunks, "reps": args.reps, "threshold": THR, "generated_contacts": GEN,
        "model": "synth.GCNConfig() (MF-size head)",
        "two_step_proteins_per_s": args.pairs / float(np.median(times["two_step"])),
        "fused_proteins_per_s": args.pairs / float(np.median(times["fused"])),
        "two_step_ms": [round(t * 1e3, 2) for t in times["two_step"]],
        "fused_ms": [round(t * 1e3, 2) for t in times["fused"]],
        "two_step_host_ms_median": {k: float(np.median(v)) for k, v in host.items()},
        "stage_ms_fused_chunk0": {name: round(ms, 3) for name, ms, _ in stages},
        "nw_align_stage_ms": sum(ms for name, ms, _ in stages if name == "nw_align"),
        "nw_cells_chunk0": cells,
        "max_abs_score_diff_routes": worst,
    }
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
