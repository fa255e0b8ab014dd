#!/usr/bin/env python
"""bench.py — throughput of the structure-branch hot path (contact-map build + alignment transfer + DeepFRI GCN forward) on
N B200s of one node, one process per GPU.

  python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference ...                     # the reference's CPU path (oracle) on the host cores

Workloads (`--workload`, BASELINE.json `configs[i]`):
  config4 (default)  the 1M-protein metagenomic MF job, L ~ LogNormal(median 250, sigma 0.6) clipped to [50, 1000], Markov-gapped
                     alignments, random-walk C-alpha structures, 10 A maps, random-init MF head C = 489 in the reference's
                     ONNX layout.  The job's proteins (protein i = a pure function of (seed 5, i)) are partitioned over the
                     ranks by length-balanced LPT bins (`sharding.lpt_bins`) and every rank streams its bin in chunks of
                     <= 16,384 proteins.  One timed "step" = the whole path over one chunk per GPU:
                       value  = inputs of the chunk resident in HBM, CUDA events;
                       e2e    = the chunks of the rank's bin, one per step, from PYTHON LISTS of str / ndarray through
                                `Predictor.submit_structures` / `wait` (C packing into pinned memory, H2D, kernels, D2H; two jobs
                                in flight); with N > 1 the ranks' scores land in a node-local shared, page-locked
                                result matrix (`distributed.ScoreBoard`): the host result gather is a barrier;
                     then (not a step-contract number) `sharded_job`: the whole 1M-protein job end to end, strong scaling.
  config0            1,000 proteins L~U{100..500}, MF head: one step = all 1,000 proteins.
  config1            contact-map build + alignment transfer only, 100k pairs at 6 A: one step = one chunk of 16,384 pairs;
                     metric pairs/s; roofline against HBM for both output layouts (bit-packed, and the reference's dense int32).
  config2            the four heads (MF, BP, CC, EC) on 10k proteins (maps and LM shared): one step = all heads on all proteins.
  config3            2,000 proteins L 1000-2500: one step = all of them.

Prints ONE JSON line on rank 0 (contract in the task statement).
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
WORKLOAD_NAMES = ("config0", "config1", "config2", "config3", "config4")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config4", choices=WORKLOAD_NAMES)
    ap.add_argument("--proteins", type=int, default=0, help="proteins per chunk (0 = the workload's default)")
    ap.add_argument("--job-proteins", type=int, default=-1,
                    help="config4: size of the sharded job (default 1,000,000; 0 skips the sharded_job leg)")
    ap.add_argument("--engine", default="auto", choices=["auto", "simt", "tc"])
    ap.add_argument("--cpu-sample", type=int, default=400, help="proteins (pairs) in the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (rank 0): the GO-term "
                         "scores of the resident leg; config2: every head's scores from the end-to-end leg; config1: the "
                         "bit-packed contact maps of the end-to-end leg.  Outputs above 64 MB in all are a fixed, seeded sample")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


ARGS = parse()
if ARGS.impl == "reference":
    # the CPU arm uses every host core; torch.distributed.run exports OMP_NUM_THREADS=1 to its workers, which would otherwise
    # pin the BLAS / OpenMP pools of this process to one thread
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[k] = str(os.cpu_count() or 1)

import statistics  # noqa: E402
import subprocess  # noqa: E402
import tempfile  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))      # the CPU arm (cpu_baseline / --impl reference) is the only user
import mdf_pkg  # noqa: E402

mdf_pkg.load()
from metagenomic_deepfri_b200 import synth  # noqa: E402

GEN = 2
HEADS = {"mf": 489, "bp": 1943, "cc": 320, "ec": 538}
CHUNK = 16384
DESCRIPTIONS = {
    "config4": "BASELINE configs[4]: metagenomic MF job, L~LogNormal(250, 0.6) clipped [50,1000], protein i keyed by (seed 5, i), LPT bins "
               "over the ranks, chunks of <= {n} proteins per GPU per step; gapped alignments, 10A maps, MF head C=489",
    "config0": "BASELINE configs[0]: {n} synthetic proteins L~U{{100..500}}, gapped alignments, 10A maps, MF head C=489",
    "config1": "BASELINE configs[1]: contact-map build + alignment transfer only, chunks of {n} of 100,000 query/target pairs "
               "(L~U{{50..1000}}, Markov-gapped alignments, 6A, generated contacts 2)",
    "config2": "BASELINE configs[2]: MF, BP, CC and EC heads on {n} proteins, L~LogNormal(250, 0.6) clipped [50,1000], maps + LM shared",
    "config3": "BASELINE configs[3]: {n} proteins L~U{{1000..2500}}, 10A maps, MF head C=489",
}
THRESHOLDS = {"config0": 10.0, "config1": 6.0, "config2": 10.0, "config3": 10.0, "config4": 10.0}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "tflops_burst": d["bf16_tflops"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "tflops_burst": 1590.0, "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic(stage):
    """dram bytes (read + write) per launch of the stage's kernel from the committed `ncu --set full` capture of this
    same command (profiles/ncu_traffic.json, written by tools/ncu_summary.py), or None."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get(stage)
    return None


DUMP_BYTES = 60 << 20          # --dump-outputs: data bytes of all files together (< 64 MB with the .npy headers)


def dump_outputs(out_dir, scores=None, maps=None):
    """--dump-outputs.  `scores`: {name: float32 [n, C]} with a common n, written whole or as the same seeded sample of rows
    (rows.npy) when larger than DUMP_BYTES.  `maps`: bit-packed uint32 [Lq, words] per pair, a seeded sample of pairs
    written as float64 (exact for uint32): cmap_words.npy = their words, concatenated; cmap_pairs.npy = (pair, Lq) rows."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    if maps is not None:
        order = rng.permutation(len(maps))
        size = np.cumsum([maps[i].size * 8 + 16 for i in order])
        keep = np.sort(order[size <= DUMP_BYTES])
        out = {"cmap_words": np.concatenate([maps[i].ravel() for i in keep]).astype(np.float64),
               "cmap_pairs": np.array([(i, maps[i].shape[0]) for i in keep], np.float64).reshape(-1, 2)}
    else:
        n = len(next(iter(scores.values())))
        row_bytes = sum(s.shape[1] * 4 for s in scores.values())
        k = min(n, DUMP_BYTES // (row_bytes + 8))
        rows = np.arange(n) if k == n else np.sort(rng.choice(n, k, replace=False))
        out = {name: np.ascontiguousarray(s[rows], np.float32) for name, s in scores.items()}
        if k < n:
            out["rows"] = rows.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def sub(wl, idx):
    return synth.Workload([wl.query_seqs[i] for i in idx], [wl.gapped_query[i] for i in idx], [wl.gapped_target[i] for i in idx],
                          [wl.coords[i] for i in idx], wl.threshold, wl.generated_contacts, wl.name)


# ------------------------------------------------------------------------------------------ workloads
def small_workload(name, n_override):
    """configs[0..3] -> (list of chunks, description).  Same seeds as synth.config_workload."""
    idx = int(name[-1])
    full = {0: 1000, 1: 100_000, 2: 10_000, 3: 2000}[idx]
    if idx == 1:
        n = n_override or CHUNK
        wl = synth.config_workload(1, min(1.0, 4 * n / full))          # four different chunks are enough for the step loop
        chunks = [sub(wl, range(lo, min(len(wl), lo + n))) for lo in range(0, len(wl), n)]
        return chunks, DESCRIPTIONS[name].format(n=n)
    n = n_override or full
    wl = synth.config_workload(idx, n / full)
    return [wl], DESCRIPTIONS[name].format(n=len(wl))


def config4_plan(args, world):
    """Lengths of the whole job, LPT bins, chunks: identical on every rank (pure function of the seed)."""
    from metagenomic_deepfri_b200 import distributed, sharding
    n_chunk = args.proteins or CHUNK
    job_n = 1_000_000 if args.job_proteins < 0 else args.job_proteins
    # the step legs need at least `chunks_wanted` chunks per rank even when the sharded_job leg is off or small
    plan_n = max(job_n, world * n_chunk * 2)
    lengths = synth.keyed_lengths(np.arange(plan_n), 5)
    shards = distributed.shard_job(lengths, world, max_proteins=n_chunk)
    bins = [np.concatenate(s) if s else np.zeros(0, np.int64) for s in shards]
    pred_imb = sharding.imbalance(bins, lengths)
    return lengths, shards, job_n, plan_n, pred_imb


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_predictor(model_path):
    """The GCN half of the CPU arm: the `.onnx` file executed on PyTorch's CPU kernels (oracle/torch_ref.py: torch.nn.LSTM
    / oneDNN GEMMs - the fastest stand-in for onnxruntime this image has; onnxruntime itself is absent), batch = 1 per call
    like pipeline.py:301-319, all host threads."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch
    import torch_ref
    torch.set_num_threads(os.cpu_count() or 1)
    return torch_ref.Predictor(model_path), torch.get_num_threads()


def cpu_cmap(wl, i, thr):
    import cmap_oracle as co
    ref = co.ref_module()
    if ref is not None:
        D = ref.pairwise_sqeuclidean(wl.coords[i])
        sp = np.argwhere((D < thr ** 2).astype(np.int32) == 1).astype(np.int32)        # bio_utils.py:220-223
        return ref.align_contact_map(wl.gapped_query[i], wl.gapped_target[i], sp, GEN)
    return co.build_align_contact_map(wl.gapped_query[i], wl.gapped_target[i], wl.coords[i], thr, GEN)


_POOL_WL = None


def _pool_cmap(args):
    i, thr = args
    return cpu_cmap(_POOL_WL, i, thr).shape[0]


def cpu_path(wl, thr, idx, model_paths, pool=None):
    """The reference's CPU path on proteins `idx`: compiled contact_map_utils.pyx (oracle/_ref; the C port when it is not
    built) + the NumPy glue of bio_utils.py:214-223, then one forward_pass per protein and head.  -> (units/s, seconds, cores, what)"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import cmap_oracle as co
    cm_impl = "reference contact_map_utils.pyx" if co.ref_module() is not None else "C port"
    if not model_paths:                               # configs[1]: maps only, a process pool like pipeline.py:476-481
        t0 = time.perf_counter()
        if pool is not None:
            pool.map(_pool_cmap, [(int(i), thr) for i in idx], chunksize=4)
        else:
            for i in idx:
                cpu_cmap(wl, int(i), thr)
        dt = time.perf_counter() - t0
        return len(idx) / dt, dt, (pool._processes if pool is not None else 1), f"cmap: {cm_impl}, process pool"
    preds, threads = [], 1
    for p in model_paths:
        pr, threads = cpu_predictor(p)
        preds.append(pr)
    t0 = time.perf_counter()
    for i in idx:
        cm = cpu_cmap(wl, int(i), thr)
        for pr in preds:
            pr.forward_pass(wl.query_seqs[int(i)], cm)
    dt = time.perf_counter() - t0
    return len(idx) / dt, dt, threads, (f"cmap: {cm_impl}; GCN: torch-CPU executor of the .onnx file standing in for onnxruntime "
                                       f"({threads} threads), batch=1 per call")


def write_models(tmp, workload):
    if workload == "config1":
        p = os.path.join(tmp, "mf.onnx")
        synth.write_gcn_model(p, synth.GCNConfig())
        return {"mf": p}
    heads = HEADS if workload == "config2" else {"mf": 489}
    out = {}
    for h, C in heads.items():
        out[h] = os.path.join(tmp, f"{h}.onnx")
        synth.write_gcn_model(out[h], synth.GCNConfig(n_terms=C), seed=1234 if h == "mf" else 77 + C)
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    global _POOL_WL
    thr = THRESHOLDS[args.workload]
    if args.workload == "config4":
        n = args.proteins or CHUNK
        wl, workload = synth.keyed_workload_parallel(np.arange(2048), 5, min(8, os.cpu_count() or 1)), DESCRIPTIONS["config4"].format(n=n)
    else:
        chunks, workload = small_workload(args.workload, min(args.proteins or 2048, 2048) if args.workload == "config1" else args.proteins)
        wl = chunks[0]
    maps_only = args.workload == "config1"
    per_step = 64 if maps_only else (2 if args.workload in ("config2", "config3") else 6)
    pool = None
    if maps_only:
        import multiprocessing as mp
        _POOL_WL = wl
        pool = mp.get_context("fork").Pool(os.cpu_count() or 1)
    with tempfile.TemporaryDirectory() as d:
        models = [] if maps_only else list(write_models(d, args.workload).values())
        rng = np.random.default_rng(0)
        times, cores, what = [], 1, ""
        for s in range(args.warmup + args.steps):
            idx = rng.choice(len(wl), min(per_step, len(wl)), replace=False)
            _, dt, cores, what = cpu_path(wl, thr, idx, models, pool)
            if s >= args.warmup:
                times.append(dt)
    if pool is not None:
        pool.close()
    total = sum(times)
    value = per_step * args.steps / total
    unit = "pairs/s" if maps_only else "proteins/s"
    line = {
        "impl": "reference", "metric": metric_name(args.workload), "value": value, "unit": unit,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "sample": f"{per_step} units per step drawn from {len(wl)} of the workload's proteins", "cpu_path": what},
        "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": "port",
                         "sample": f"{per_step * args.steps} units; {what}; host has {os.cpu_count()} cpus"},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def metric_name(workload):
    return {"config1": "pairs/sec (contact-map build + alignment transfer)",
            "config2": "proteins/sec (GCN MF+BP+CC+EC fwd incl. cmap)"}.get(workload, "proteins/sec (GCN MF fwd incl. cmap)")


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ B200 arm
def prepare_inputs(args, rank, world):
    """Host-side inputs of this rank.  Runs before the process group and CUDA exist: the generators fork worker processes."""
    global _POOL_WL
    thr = THRESHOLDS[args.workload]
    maps_only = args.workload == "config1"
    t_gen = time.perf_counter()
    sharded = None
    if args.workload == "config4":
        lengths, shards, job_n, plan_n, pred_imb = config4_plan(args, world)
        my_chunks_idx = shards[rank]
        chunks_wanted = len(my_chunks_idx) if job_n else min(len(my_chunks_idx), 2)
        procs = max(1, min(16, (os.cpu_count() or 1) // max(1, min(world, 8))))
        ids = np.concatenate(my_chunks_idx[:chunks_wanted])
        wl_all = synth.keyed_workload_parallel(ids, 5, procs, threshold=thr)
        chunks, lo = [], 0
        for ci in my_chunks_idx[:chunks_wanted]:
            chunks.append(sub(wl_all, range(lo, lo + len(ci))))
            lo += len(ci)
        del wl_all
        workload = DESCRIPTIONS["config4"].format(n=args.proteins or CHUNK)
        sharded = dict(job_n=job_n, lengths=lengths, my_idx=my_chunks_idx, pred_imb=pred_imb)
    else:
        chunks, workload = small_workload(args.workload, args.proteins)
    gen_s = time.perf_counter() - t_gen
    cpu_pool = None
    if maps_only and rank == 0 and world == 1 and not args.no_cpu_baseline:
        import multiprocessing as mp
        _POOL_WL = chunks[0]
        cpu_pool = mp.get_context("fork").Pool(os.cpu_count() or 1)      # forked before the CUDA context exists
    return dict(chunks=chunks, workload=workload, sharded=sharded, gen_s=gen_s, cpu_pool=cpu_pool)


def run_b200(args, rank, world, local_rank, inputs):
    thr = THRESHOLDS[args.workload]
    maps_only = args.workload == "config1"
    multi_head = args.workload == "config2"
    chunks, workload, sharded, gen_s, cpu_pool = (inputs[k] for k in ("chunks", "workload", "sharded", "gen_s", "cpu_pool"))

    import torch
    import torch.distributed as dist
    from metagenomic_deepfri_b200 import _lib, bio_utils, distributed, pipeline, predict
    torch.cuda.set_device(local_rank)
    stream = torch.cuda.Stream()             # a real (non-NULL) stream shared by torch and the library
    torch.cuda.set_stream(stream)
    ctx = _lib.Context(local_rank, stream=stream.cuda_stream)
    tmp = tempfile.mkdtemp()
    models = write_models(tmp, args.workload)
    preds = {h: predict.Predictor(p, context=ctx) for h, p in models.items()}
    pred = preds["mf"]
    if args.engine != "auto":
        for p in preds.values():
            p.set_engine(args.engine)
    C = sum(p.n_terms for p in preds.values()) if multi_head else pred.n_terms

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allsum(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t[0])

    def allmax(*xs):
        t = torch.tensor([float(x) for x in xs], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")     # > 126 MB L2
    wl0 = chunks[0]
    n0 = len(wl0)
    T0 = sum(len(s) for s in wl0.query_seqs)

    def run_resident(batch):
        if maps_only:
            pred.run(batch, thr, GEN, upto=1)
        elif multi_head:
            batch.invalidate()                  # nothing computed by an earlier step may be reused: every step builds the maps and runs the LM
            for p in preds.values():
                p.run(batch, thr, GEN, share=True)      # within the step the four heads share maps + LM output (pipeline.py:546-655)
        else:
            pred.run(batch, thr, GEN)

    # ---- resident leg: inputs already in HBM when the timed region starts
    batch = pred.upload(wl0.query_seqs, wl0.gapped_query, wl0.gapped_target, wl0.coords)
    for _ in range(args.warmup):
        run_resident(batch)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    ctx.profile(True)                           # per-stage CUDA events on the launch stream, inside the timed steps (roofline object)
    for s in range(args.steps):
        flush.zero_()                           # L2 flush between timed iterations (outside the events)
        ev[s][0].record(stream)
        run_resident(batch)
        ev[s][1].record(stream)
    barrier()
    timed_stages = ctx.profile_report()
    ctx.profile(False)
    launches = ctx.launch_count - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    dense = None
    if maps_only:                               # the reference-layout (dense int32) output of the same maps: HBM-bound variant
        for _ in range(2):
            cells = pred.unpack_dense(batch)
        ctx.profile(True)
        for _ in range(max(3, args.steps)):
            flush.zero_()
            pred.unpack_dense(batch)
        rep = [r for r in ctx.profile_report() if r[0] == "cmap_unpack_dense"]
        ctx.profile(False)
        dms = sum(r[1] for r in rep) / len(rep)
        dense = {"cells": cells, "unpack_ms": dms, "bytes": rep[0][2]}
    # (the batch holds the scores of the head that ran last)
    scores_resident = None if maps_only else list(preds.values())[-1].fetch_scores(batch)
    batch.close()
    del batch

    # ---- end-to-end leg: Python lists -> (C packing into pinned memory) -> H2D -> path -> D2H, through the public calls
    class Aln:
        def __init__(self, w, i):
            self.query_name, self.target_name = f"q{i}", f"t{i}"
            self.gapped_sequence, self.gapped_target, self.coords = w.gapped_query[i], w.gapped_target[i], w.coords[i]
            self.query_sequence = w.query_seqs[i]
    steps_chunks = [chunks[s % len(chunks)] for s in range(args.steps)]
    n_e2e = sum(len(c) for c in steps_chunks)
    h2d = d2h = 0
    if maps_only:
        aln_chunks = [[Aln(c, i) for i in range(len(c))] for c in chunks]
        # the maps of one step (0.8 GB) land in a page-locked arena that is reused from step to step (`out=`): into fresh pageable
        # arrays the device -> host copy is staged and page-faults its destination, which cost more than everything else together
        words = max(int(sum(len(q) * ((len(q) + 127) // 128 * 4) for q in c.query_seqs)) for c in chunks)
        arena = torch.empty(words, dtype=torch.int32, pin_memory=True).numpy().view(np.uint32)
        for _ in range(max(1, args.warmup)):
            bio_utils.build_align_contact_maps(aln_chunks[0], thr, GEN, packed=True, out=arena)
        barrier()
        t0 = time.perf_counter()
        for s in range(args.steps):
            maps = bio_utils.build_align_contact_maps(aln_chunks[s % len(chunks)], thr, GEN, packed=True, out=arena)
        barrier()
        e2e_s = time.perf_counter() - t0
        c = steps_chunks[0]
        h2d = int(sum(x.nbytes for x in c.coords) + 2 * sum(len(q) for q in c.gapped_query))
        d2h = int(sum(m.nbytes for m in maps))
    elif multi_head:
        alns = [Aln(wl0, i) for i in range(n0)]
        for _ in range(max(1, args.warmup)):
            pipeline.predict_structures(preds, alns, thr, GEN)
        barrier()
        t0 = time.perf_counter()
        for s in range(args.steps):
            out_heads, _, _ = pipeline.predict_structures(preds, alns, thr, GEN)
        barrier()
        e2e_s = time.perf_counter() - t0
        local_scores = np.concatenate([out_heads[h] for h in preds], axis=1)
        assert np.abs(out_heads[list(preds)[-1]] - scores_resident).max() < 1e-5, "resident and end-to-end legs disagree"
        h2d = int(sum(x.nbytes for x in wl0.coords) + 2 * sum(len(q) for q in wl0.gapped_query) + T0)
        d2h = int(local_scores.nbytes)
    else:
        out_host = torch.empty((n_e2e, C), dtype=torch.float32, pin_memory=True).numpy()

        def submit(c, rows):
            return pred.submit_structures(c.query_seqs, c.gapped_query, c.gapped_target, c.coords, thr, GEN, out=rows)
        for _ in range(max(1, args.warmup)):
            distributed.stream_chunks(submit, [(chunks[0], n0)], out_host[:n0])
        board = all_scores = None
        if world > 1:
            # host result gather without a collective: the result matrix of all ranks lives in node-local shared memory, page-locked
            # in every rank (distributed.ScoreBoard); each rank's device -> host copies land directly in its row range and the
            # "gather" is the barrier after the last chunk.  (An NCCL gather + ONE 2.5 GB device -> host copy on rank 0 cost 11 %
            # of the 8-GPU end-to-end time.)
            counts = np.zeros(world + 1, np.int64)
            tcount = torch.tensor([n_e2e], dtype=torch.int64, device="cuda")
            lst = [torch.zeros_like(tcount) for _ in range(world)]
            dist.all_gather(lst, tcount)
            counts[1:] = np.cumsum([int(x.item()) for x in lst])
            gatherer = my_rows = None
            try:
                board = distributed.ScoreBoard(int(counts[-1]), C)
                out_host = board.rows(int(counts[rank]), int(counts[rank + 1]))
                distributed.stream_chunks(submit, [(chunks[0], n0)], out_host[:n0])      # warm-up into the shared rows
            except RuntimeError:        # (agreed on by all ranks) no usable /dev/shm: one NCCL gather at the end instead
                board = None
                gatherer = distributed.ScoreGather(n_e2e, int(counts[-1]), C)
                my_rows = np.arange(counts[rank], counts[rank + 1])
                gatherer.gather(my_rows, out_host)                  # warm-up: NCCL builds its gather channels lazily
        barrier()
        t0 = time.perf_counter()
        distributed.stream_chunks(submit, [(c, len(c)) for c in steps_chunks], out_host)
        local_scores = out_host
        if world > 1:       # scores of every step of every rank are now readable on rank 0
            all_scores = board.finish() if board is not None else gatherer.gather(my_rows, local_scores)
            if rank == 0:
                assert all_scores.shape == (int(counts[-1]), C)
        barrier()
        e2e_s = time.perf_counter() - t0
        c = steps_chunks[0]
        h2d = int(sum(x.nbytes for x in c.coords) + 2 * sum(len(q) for q in c.gapped_query) + sum(len(q) for q in c.query_seqs))
        d2h = int(len(c) * C * 4)
        if len(chunks) == 1 or args.steps >= 1:
            assert np.abs(local_scores[:n0] - scores_resident).max() < 1e-5, "resident and end-to-end legs disagree"
        if board is not None:
            local_scores = out_host = all_scores = None
            board.close()
    clocks = sampler.stop() if rank == 0 else None

    # ---- config4: the whole sharded job, end to end (strong scaling): every rank streams ALL chunks of its LPT bin from Python
    # lists, rank 0 gathers the [job_n, C] score matrix in protein order
    job = None
    if sharded and sharded["job_n"] > 0:
        my_idx = [ci[ci < sharded["job_n"]] for ci in sharded["my_idx"]]
        my_chunks = [(sub(c, range(len(ix))) if len(ix) != len(c) else c) for c, ix in zip(chunks, my_idx) if len(ix)]
        my_ids = np.concatenate([ix for ix in my_idx if len(ix)]) if my_chunks else np.zeros(0, np.int64)
        job_out = torch.empty((len(my_ids), C), dtype=torch.float32, pin_memory=True).numpy()

        def submit(c, rows):
            return pred.submit_structures(c.query_seqs, c.gapped_query, c.gapped_target, c.coords, thr, GEN, out=rows)
        chunk_ids = [ix for ix in my_idx if len(ix)]
        job_board = job_gather = on_done = None
        if world > 1:
            # result matrix in protein order: shared, page-locked, allocated before the clock starts; every rank scatters a chunk's
            # rows into it while the next chunks compute
            try:
                job_board = distributed.ScoreBoard(sharded["job_n"], C)
                on_done = lambda k, rows: job_board.put(chunk_ids[k], rows)         # noqa: E731
            except RuntimeError:
                job_board = None
        if job_board is None:
            job_gather = distributed.ScoreGather(len(my_ids), sharded["job_n"], C)
        result_gather = ("none (one rank)" if world == 1 else
                         "NCCL gather + one device->host copy on rank 0" if job_board is None else
                         "node-local shared result matrix (%s), rows scattered per chunk, barrier" %
                         ("page-locked" if job_board._registered else "pageable"))
        barrier()
        t0 = time.perf_counter()
        distributed.stream_chunks(submit, [(c, len(c)) for c in my_chunks], job_out, on_done=on_done)
        t_rank = time.perf_counter() - t0
        final = job_board.finish() if job_board is not None else job_gather.gather(my_ids, job_out)
        barrier()
        job_s = time.perf_counter() - t0
        busy = allsum(t_rank) / world
        job_s, t_rank_max = allmax(job_s, t_rank)
        if rank == 0:
            assert final is not None and final.shape == (sharded["job_n"], C) and np.isfinite(final[::997]).all()
            assert np.abs(final[my_ids[:64]] - job_out[:64]).max() == 0.0
        if job_board is not None:
            final = None
            job_board.close()
        job = {"proteins": sharded["job_n"], "residues": int(sharded["lengths"][:sharded["job_n"]].sum()), "seconds": job_s,
               "proteins_per_s": sharded["job_n"] / job_s, "scaling": "strong",
               "chunks_per_rank": len(my_chunks), "imbalance_measured": t_rank_max / busy if busy else None,
               "imbalance_predicted_lpt": sharded["pred_imb"], "gather_and_tail_s": job_s - t_rank_max,
               "input": "Python lists of str / ndarray per protein -> Predictor.submit_structures (two jobs in flight)",
               "result_gather": result_gather, "generator_s": round(gen_s, 1)}

    # max over ranks
    dev_ms, e2e_ms = allmax(dev_ms, e2e_s * 1e3)
    units_resident = allsum(n0 * args.steps)
    units_e2e = allsum(n_e2e)

    # ---- per-stage profile for the roofline object: the stage events recorded live inside the timed steps, averaged per step
    PROF_PASSES = max(1, args.steps)
    agg = {}
    for name, ms, units in timed_stages:
        a = agg.setdefault(name, [0.0, 0.0, 0])
        a[0] += ms / PROF_PASSES; a[1] += units / PROF_PASSES; a[2] += 1
    for a in agg.values():
        a[2] //= PROF_PASSES
    peaks = measured_peaks()
    stage_total = sum(a[0] for a in agg.values())
    dname, (dms, dunits, dcount) = max(agg.items(), key=lambda kv: kv[1][0])
    if dname == "cmap_build_transfer":
        roof = {"bound": "hbm", "achieved": dunits / (dms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s"}
    else:
        roof = {"bound": "tensor", "achieved": dunits / (dms * 1e-3) / 1e12, "peak": peaks["tflops"], "unit": "TFLOP/s"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["traffic"] = ncu_traffic(dname + "_config1" if maps_only else dname) or ncu_traffic(dname)
    roof["kernel"] = dname
    roof["launches_per_step"] = dcount
    roof["share_of_step"] = dms / stage_total if stage_total else None
    roof["peak_source"] = peaks["source"] + (" sustained bf16" if roof["bound"] == "tensor" else "")
    roof["stages_ms"] = {k: round(v[0], 4) for k, v in agg.items()}
    if maps_only:
        lq = np.array([len(s) for s in wl0.query_seqs], np.float64)
        flops = float((9 * lq * (lq - 1) / 2).sum())            # SURVEY 8d: 9 non-fusable FP32 ops per unordered residue pair
        roof["fp32_issue"] = {"achieved_Tops": flops / (dms * 1e-3) / 1e12, "peak_Tops": 37.0, "frac": flops / (dms * 1e-3) / 1e12 / 37.0,
                              "note": "bit-packed output makes the kernel FP32-issue-bound, not HBM-bound (SURVEY 8d)"}
        roof["dense_output_variant"] = {"kernel": "unpack_dense_kernel", "bound": "hbm", "bytes_per_launch": dense["bytes"],
                                        "ms": dense["unpack_ms"], "achieved": dense["bytes"] / (dense["unpack_ms"] * 1e-3) / 1e9,
                                        "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                        "frac": dense["bytes"] / (dense["unpack_ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                        "note": "reference layout: int32 [Lq, Lq] per pair written to HBM (4 bytes per cell)"}

    if rank != 0:
        return
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        idx = np.random.default_rng(0).choice(n0, min(args.cpu_sample if not multi_head else max(8, args.cpu_sample // 8), n0), replace=False)
        pps, dt, cores, what = cpu_path(wl0, thr, idx, [] if maps_only else list(models.values()), cpu_pool)
        if cpu_pool is not None:
            cpu_pool.close()
        cpu = {"value": pps, "unit": "pairs/s" if maps_only else "proteins/s", "cores": cores, "kind": "port",
               "sample": f"{len(idx)} of the {n0} units of one step ({dt:.1f} s); {what}; host has {os.cpu_count()} cpus"}
    unit = "pairs/s" if maps_only else "proteins/s"
    line = {
        "metric": metric_name(args.workload), "value": units_resident / (dev_ms * 1e-3), "unit": unit,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if maps_only or pred.engine == "simt" else "f16 (hi/lo split weights) with f32 accumulate",
        "data": "synthetic",
        "config": {"workload": workload, "units_per_step_per_gpu": n0, "residues_per_step_per_gpu": T0,
                   "threshold_A": thr, "generated_contacts": GEN, "engine": "cmap kernels" if maps_only else pred.engine,
                   "heads": list(preds) if not maps_only else [],
                   "l2": "flushed between timed iterations (256 MiB memset outside the event pairs)",
                   "timing": "per-step CUDA events on the launch stream, summed over steps, max over ranks",
                   "generator_s": round(gen_s, 1)},
        "e2e": {"value": units_e2e / (e2e_ms * 1e-3), "unit": unit,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / args.steps,
                "distinct_chunks": len(chunks),
                "note": ("bio_utils.build_align_contact_maps(packed=True, out=<reused page-locked arena>) from Python lists of alignments: C packing on host threads -> H2D -> fused kernels -> D2H of the bit-packed maps" if maps_only else
                         "pipeline.predict_structures from Python lists (one upload, all heads)" if multi_head else
                         "Predictor.submit_structures / wait from Python lists of str / ndarray: C packing into pinned memory -> H2D -> all "
                         "kernels -> D2H scores, two jobs in flight per GPU; N > 1: scores land in a node-local shared pinned result matrix, the gather is a barrier; wall clock")},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roof,
        "cpu_baseline": cpu,
    }
    if job:
        line["sharded_job"] = job
    if args.dump_outputs:
        if maps_only:
            dump_outputs(args.dump_outputs, maps=maps)
        else:
            dump_outputs(args.dump_outputs, {f"scores_{h}": out_heads[h] for h in preds} if multi_head else {"scores": scores_resident})
    print(json.dumps(line), flush=True)


def main():
    # stdout carries exactly ONE JSON line: libraries that print there (NCCL's version banner) are sent to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    args = ARGS
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    inputs = prepare_inputs(args, rank, world)
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, world, local_rank, inputs)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
