"""Sequence-only DeepCNN branch (SURVEY.md 8f row 2): proteins/s of `Predictor.forward_sequences` on unaligned queries with
the metagenomic length distribution of BASELINE configs[4] (L ~ LogNormal(250, 0.6) clipped to [50, 1000]) and the trained
models' shape (16 x 512 filters of widths 8..128, MF head C = 489, random-init weights in the reference's ONNX layout).

Reports: resident throughput (CUDA-event stage times from mdf_ctx_profile), the convolution kernel's tensor-pipe fraction
(algorithmic FLOPs = 2 * 26 * sum(w * F) per residue; the kernel issues 13 K-steps of 16 per 8 positions = 26 columns
per position, plus the padded rows of partly filled 128-residue tiles), end-to-end throughput through forward_sequences (host strings in,
host scores out), a parity check against the oracle on a bounded sample, and the oracle's own CPU rate.

The streamed leg runs K chunks of `--proteins` sequences from Python lists through `submit_sequences` with two jobs in flight
(`distributed.stream_chunks`, scores into page-locked memory); it alternates in the same process with the resident leg (each of
the K chunks uploaded, then its run timed) and the `forward_sequences` leg over the same K chunks, and reports the largest |score difference| against `forward_sequences` over every
timed chunk (the same kernels run on the same inputs: it must be exactly 0).  The card's name and power limit are read in the same
run (`nvidia-smi --query-gpu=name,power.limit`).

  python tools/cnn_bench.py [--proteins 16384] [--reps 5] [--chunks 8] [--cpu-sample 8] [--out profiles/cnn_bench.json]
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import mdf_pkg  # noqa: E402

mdf_pkg.load()
from metagenomic_deepfri_b200 import distributed, synth, predict, _lib  # noqa: E402
import gcn_oracle as go  # noqa: E402


def card():
    """Name and power limit of the GPU this process runs on (read-only query)."""
    import subprocess
    dev = os.environ.get("LOCAL_RANK", "0")
    r = subprocess.run(["nvidia-smi", "-i", dev, "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=60)
    name, power = [x.strip() for x in r.stdout.strip().split(",")]
    return {"gpu": name, "power_limit": power}


def configs4_lengths(rng, n):
    return np.clip(np.exp(rng.normal(np.log(250.0), 0.6, size=n)), 50, 1000).astype(np.int64)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--proteins", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cpu-sample", type=int, default=8)
    ap.add_argument("--chunks", type=int, default=8, help="K chunks of --proteins sequences in the streamed / forward_sequences legs")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    rng = np.random.default_rng(5)
    lengths = configs4_lengths(rng, args.proteins)
    seqs = synth.random_sequences(rng, lengths)
    cfg = synth.CNNConfig()
    path = os.path.join(tempfile.mkdtemp(), "DeepCNN-MERGED_mf.onnx")
    synth.write_cnn_model(path, cfg)
    pred = predict.Predictor(path)
    ctx = _lib.default_context()
    T = int(lengths.sum())
    flops = 2.0 * 26 * sum(w * f for w, f in zip(cfg.filter_lens, cfg.num_filters)) * T
    def k_blocks(w):      # K = 16 steps of a conv (csrc/cnn_tc.cu: 13 per 8 positions), four per 16 KiB weight tile
        return -(-(w + (w + 1) // 2 + ((w + 3) // 4 + 1) // 2) // 4)
    issued = 2.0 * sum(64 * k_blocks(w) * f for w, f in zip(cfg.filter_lens, cfg.num_filters)) * float(((lengths + 127) // 128 * 128).sum())
    pred.upload_sequences(seqs)
    for _ in range(2):
        pred.run_sequences()
    ctx.synchronize()
    ctx.profile(True)
    for _ in range(args.reps):
        pred.run_sequences()
    ctx.synchronize()
    rep = ctx.profile_report()
    ctx.profile(False)
    stage = {}
    for name, ms, units in rep:
        stage.setdefault(name, []).append(ms)
    conv_ms = float(np.median(stage["cnn_conv"]))
    head_ms = float(np.median(stage["cnn_head"]))
    times = []
    for _ in range(args.reps):
        ctx.synchronize()
        t0 = time.perf_counter()
        pred.run_sequences()
        ctx.synchronize()
        times.append(time.perf_counter() - t0)
    dt = float(np.median(times))
    e2e = []
    for _ in range(3):
        t0 = time.perf_counter()
        scores = pred.forward_sequences(seqs)
        e2e.append(time.perf_counter() - t0)
    # ---- K chunks from Python lists: resident / forward_sequences / streamed jobs, alternated rep by rep
    import torch
    chunks = [seqs] + [synth.random_sequences(rng, configs4_lengths(rng, args.proteins)) for _ in range(args.chunks - 1)]
    K, n = len(chunks), args.proteins
    streamed_out = torch.empty((K * n, pred.n_terms), dtype=torch.float32, pin_memory=True).numpy()
    want = np.empty_like(streamed_out)
    legs = {"resident": [], "forward_sequences": [], "streamed": []}
    worst_stream = 0.0
    pred.submit_sequences(chunks[1]).wait()            # first job: slot blocks allocated and page-locked outside the timed window
    for rep in range(args.reps):
        # the same K chunks in all three legs; the resident leg times the runs only, each chunk uploaded before its run
        resident = 0.0
        for ch in chunks:
            pred.upload_sequences(ch)
            ctx.synchronize()
            t0 = time.perf_counter()
            pred.run_sequences()
            ctx.synchronize()
            resident += time.perf_counter() - t0
        legs["resident"].append(resident)
        t0 = time.perf_counter()
        for k, ch in enumerate(chunks):
            pred.forward_sequences(ch, out=want[k * n:(k + 1) * n])
        legs["forward_sequences"].append(time.perf_counter() - t0)
        streamed_out[...] = np.nan
        t0 = time.perf_counter()
        distributed.stream_chunks(lambda k, rows: pred.submit_sequences(chunks[k], out=rows), ((k, n) for k in range(K)), streamed_out)
        legs["streamed"].append(time.perf_counter() - t0)
        worst_stream = float(np.max([worst_stream, np.abs(streamed_out - want).max()]))     # NaN (a row never written) propagates
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    peak = peaks.get("bf16_tflops_sustained", 1400.0)
    out = {"proteins": args.proteins, "residues": T, "proteins_per_s_resident": args.proteins / dt, "ms_per_batch": dt * 1e3,
           "conv_ms": conv_ms, "head_ms": head_ms, "conv_algorithmic_TFLOPs": flops / conv_ms / 1e9,
           "conv_frac_of_sustained_peak": flops / conv_ms / 1e9 / peak, "conv_issued_TFLOPs": issued / conv_ms / 1e9,
           "conv_issued_frac": issued / conv_ms / 1e9 / peak, "peak_TFLOPs": peak,
           "proteins_per_s_e2e": args.proteins / float(np.median(e2e)),
           "chunks": K, "reps": args.reps}
    for leg, ts in legs.items():
        out[f"{leg}_proteins_per_s"] = K * n / float(np.median(ts))
        out[f"{leg}_s_per_{K}_chunks"] = [round(t, 4) for t in ts]
    out["streamed_vs_forward_sequences_max_abs_diff"] = worst_stream
    out.update(card())
    # parity on a bounded sample + the oracle's CPU rate (fp32 NumPy ONNX interpreter standing in for onnxruntime)
    orc = go.Predictor(path)
    idx = np.linspace(0, args.proteins - 1, args.cpu_sample).astype(int)
    t0 = time.perf_counter()
    worst = 0.0
    for i in idx:
        worst = max(worst, float(np.abs(orc.forward_pass(seqs[i]) - scores[i]).max()))
    cpu_dt = time.perf_counter() - t0
    out["max_abs_score_error_vs_oracle"] = worst
    out["cpu_oracle_proteins_per_s"] = len(idx) / cpu_dt
    out["cpu_cores"] = os.cpu_count()
    assert worst <= 1e-3, worst
    assert worst_stream == 0.0, worst_stream
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
