"""Worker of tests/test_gpu_cnn_jobs.py::test_two_gpu_sharded_run (launched by torch.distributed.run, one process per GPU): the
sequence-only DeepCNN branch sharded on a linear cost, streamed through submit_sequences jobs into a node-local ScoreBoard; rank 0
compares the gathered matrix with forward_sequences over all sequences.  argv[1]: the DeepCNN .onnx file."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mdf_pkg  # noqa: E402

mdf_pkg.load()
from metagenomic_deepfri_b200 import distributed, predict, synth  # noqa: E402

dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
rng = np.random.default_rng(31)
lengths = np.clip(np.exp(rng.normal(np.log(250.0), 0.6, size=2500)), 50, 1000).astype(np.int64)
seqs = synth.random_sequences(rng, lengths)              # the same on every rank (same seed)
torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))      # page-locked buffers below belong to this rank's GPU
pred = predict.Predictor(sys.argv[1], device=torch.cuda.current_device())
mine = distributed.shard_job(lengths, world, max_proteins=400, max_residues=100_000, alpha=0.0)[rank]
board = distributed.ScoreBoard(len(seqs), pred.n_terms)
local = torch.empty((sum(len(c) for c in mine), pred.n_terms), dtype=torch.float32, pin_memory=True).numpy()   # jobs overlap
distributed.stream_chunks(lambda ch, rows: pred.submit_sequences([seqs[i] for i in ch], out=rows), ((c, len(c)) for c in mine),
                          local, on_done=lambda k, rows: board.put(mine[k], rows))
final = board.finish()
if rank == 0:
    assert final is not None and np.array_equal(final, pred.forward_sequences(seqs))
    print("CNN_SHARD_OK")
else:
    assert final is None
final = None
board.close()
pred.close()
dist.destroy_process_group()
