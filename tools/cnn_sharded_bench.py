"""Sequence-only DeepCNN branch sharded across GPUs: 1M keyed sequences (protein i has the i-th length of one seeded draw of the
BASELINE configs[4] distribution, L ~ LogNormal(250, 0.6) in [50, 1000]) through `distributed.shard_job` on a linear cost
(`alpha=0`: the convolution works per residue tile) -> `stream_chunks` of `Predictor.submit_sequences` jobs, two in flight per GPU
-> a node-local `ScoreBoard`, one process per GPU.  Model: the trained models' shape (16 x 512 filters of widths 8..128, MF head
C = 489), random-init weights.

Reports per GPU count: proteins/s and job time (first rank past the start barrier to the last rank's ScoreBoard write, the
final barrier included), each rank's busy time, the residue imbalance of the LPT bins (max / mean) and the measured time
imbalance of the ranks; the name and power limit of every rank's card (`nvidia-smi --query-gpu=name,power.limit`).  Rank 0 also
checks its first chunk against `forward_sequences` (exact equality).  Sequences are generated per rank for its own bin before the
timed window.

  python tools/cnn_sharded_bench.py [--gpus 1,2,4,8] [--proteins 1000000] [--out profiles/cnn_sharded_bench.json]

launches `torch.distributed.run` once per GPU count that the machine has (counts above the visible devices are skipped and
listed as such).
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
sys.path.insert(0, os.path.join(ROOT, "tools"))
SEED = 5


def worker(args):
    import mdf_pkg
    mdf_pkg.load()
    import torch.distributed as dist
    from metagenomic_deepfri_b200 import distributed, predict, synth
    from cnn_bench import card, configs4_lengths
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    lengths = configs4_lengths(np.random.default_rng(SEED), args.proteins)
    mine = distributed.shard_job(lengths, world, alpha=0.0)[rank]
    loads = [int(lengths[np.concatenate(c)].sum()) if c else 0 for c in distributed.shard_job(lengths, world, alpha=0.0)]
    seqs = {}
    rng = np.random.default_rng([SEED, rank])
    for c in mine:
        for i, s in zip(c.tolist(), synth.random_sequences(rng, lengths[c])):
            seqs[i] = s
    chunk_seqs = [[seqs[i] for i in c.tolist()] for c in mine]
    path = os.path.join(tempfile.mkdtemp(), "DeepCNN-MERGED_mf.onnx")
    synth.write_cnn_model(path, synth.CNNConfig())
    import torch
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))    # the page-locked rows below belong to this rank's GPU
    pred = predict.Predictor(path, device=torch.cuda.current_device())
    try:
        board = distributed.ScoreBoard(args.proteins, pred.n_terms)
    except RuntimeError as e:
        print(f"rank {rank}: {e}", file=sys.stderr)
        raise
    # warm-up outside the timed window: module load, both slots' blocks allocated and page-locked at the chunk size
    warm = chunk_seqs[0]
    j1, j2 = pred.submit_sequences(warm), pred.submit_sequences(warm)
    first = j1.wait()
    j2.wait()
    check = float(np.abs(first - pred.forward_sequences(warm)).max()) if rank == 0 else 0.0
    # page-locked: a D2H copy into pageable memory would block every submit
    local = torch.empty((sum(len(c) for c in mine), pred.n_terms), dtype=torch.float32, pin_memory=True).numpy()
    dist.barrier()
    t0 = time.perf_counter()
    distributed.stream_chunks(lambda k, rows: pred.submit_sequences(chunk_seqs[k], out=rows), ((k, len(c)) for k, c in enumerate(mine)),
                              local, on_done=lambda k, rows: board.put(mine[k], rows))
    busy = time.perf_counter() - t0
    board.finish()
    job = time.perf_counter() - t0
    info = {"rank": rank, "busy_s": busy, "job_s": job, "chunks": len(mine), "proteins": int(sum(len(c) for c in mine)), **card()}
    infos = [None] * world
    dist.all_gather_object(infos, info)
    if rank == 0:
        final = board.array
        covered = bool(np.all(final[np.concatenate(mine)] == local)) if mine else True
        busy_all = [x["busy_s"] for x in infos]
        res = {"gpus": world, "proteins": args.proteins, "residues": int(lengths.sum()),
               "proteins_per_s": args.proteins / max(x["job_s"] for x in infos), "job_s": max(x["job_s"] for x in infos),
               "rank_busy_s": busy_all, "time_imbalance": max(busy_all) / float(np.mean(busy_all)),
               "residue_imbalance": max(loads) / float(np.mean(loads)), "chunks_per_rank": [x["chunks"] for x in infos],
               "first_chunk_max_abs_diff_vs_forward_sequences": check, "rank0_rows_in_scoreboard": covered,
               "cards": [{"rank": x["rank"], "gpu": x["gpu"], "power_limit": x["power_limit"]} for x in infos]}
        print("RESULT " + json.dumps(res), flush=True)
    board.close()
    pred.close()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--proteins", type=int, default=1_000_000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cnn_sharded_bench.json"))
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    import torch
    have = torch.cuda.device_count()
    runs, skipped = [], []
    for g in [int(x) for x in args.gpus.split(",")]:
        if g > have:
            skipped.append(g)
            continue
        port = str(29650 + g)
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={g}", "--master-addr",
                            "127.0.0.1", "--master-port", port, os.path.abspath(__file__), "--worker", "--proteins", str(args.proteins)],
                           capture_output=True, text=True, timeout=1800)
        lines = [ln[7:] for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
        if r.returncode != 0 or not lines:
            sys.stderr.write(r.stdout[-3000:] + r.stderr[-5000:])
            raise SystemExit(f"{g} GPU run failed (exit {r.returncode})")
        res = json.loads(lines[-1])
        print(json.dumps(res), flush=True)
        runs.append(res)
    out = {"runs": runs, "skipped_gpu_counts": skipped, "visible_gpus": have}
    if skipped:
        # not measured: the residue balance of the LPT bins those counts would run, computed on the host
        import mdf_pkg
        mdf_pkg.load()
        from metagenomic_deepfri_b200 import distributed
        from cnn_bench import configs4_lengths
        lengths = configs4_lengths(np.random.default_rng(SEED), args.proteins)
        out["lpt_residue_imbalance_host_only"] = {
            str(g): max(ls) / float(np.mean(ls)) for g in skipped
            for ls in [[int(lengths[np.concatenate(c)].sum()) for c in distributed.shard_job(lengths, g, alpha=0.0)]]}
    if runs and runs[0]["gpus"] == 1:
        base = runs[0]["proteins_per_s"]
        for r in runs:
            r["scaling_vs_1_gpu"] = r["proteins_per_s"] / base
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
