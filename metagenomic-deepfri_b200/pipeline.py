"""Batched drop-in for the GCN half of `mDeepFRI.pipeline` (`pipeline.py:292-319`, `:476-481`, `:546-655`).

The reference builds one contact map per alignment in a `multiprocessing.Pool`, then, mode by mode
(MF / BP / CC / EC), creates a `Predictor` and calls `forward_pass` once per protein, writing one TSV
row per call.  Here the same rows come out of a few batched launches:

* `run_prediction_loop` keeps the reference helper's signature and row format for callers that already
  hold `(alignment, aligned_cmap)` pairs;
* `predict_structures` is the fast path: alignments in, one score matrix per mode out.  A chunk of
  proteins is uploaded once; the contact maps are built once; the LSTM language model - identical in all
  four heads - runs once, and every further head only runs its embedding, GraphConv stack and classifier.
* `predict_pairs` does the same from (query, best-hit target, target coordinates) pairs: the alignment step
  (`align_mmseqs_results`, `alignment.py:266-322`) runs on the device once per chunk and its traceback builds the
  contact-map input directly, so no alignment string or gapped sequence passes through Python.

Nothing here falls back to the CPU; sequences without structure (`alignment.coords is None`,
`bio_utils.py:381-383`) are reported back so the caller can route them to the sequence-only branch
(`run_prediction_loop(..., net_type="cnn")` over a `DeepCNN-MERGED_*` Predictor, which streams its chunks through
`Predictor.submit_sequences`).
"""
from __future__ import annotations

import csv
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from .batching import pack_bits
from .distributed import stream_chunks
from .predict import Predictor

#: proteins per upload are bounded by residues so that the workspace stays within a few tens of GB
DEFAULT_MAX_RESIDUES = 5_000_000


def _chunks(lengths: Sequence[int], max_residues: int) -> List[Tuple[int, int]]:
    out, start, acc = [], 0, 0
    for i, L in enumerate(lengths):
        if i > start and acc + L > max_residues:
            out.append((start, i))
            start, acc = i, 0
        acc += L
    if start < len(lengths):
        out.append((start, len(lengths)))
    return out


def run_prediction_loop(predictor: Predictor, data_iterable: Iterable, data_len: int, net_type: str,
                        tsv_writer: "csv.writer", description: str = "", max_residues: int = DEFAULT_MAX_RESIDUES) -> None:
    """`pipeline._run_prediction_loop` (`pipeline.py:292-319`): one `[query_id, net_type] + scores` row per
    item, in input order.  `net_type == "gcn"` items are `(alignment, aligned_cmap)` pairs; the maps are
    bit-packed on the host and pushed through `Predictor.forward_batch` chunk by chunk."""
    items = list(data_iterable)
    if net_type == "cnn":
        # items are (query_id, sequence) pairs (`pipeline.py:313-316`): the sequence-only DeepCNN branch, two chunks in flight so
        # that the next chunk's packing and copies overlap this chunk's kernels; rows are written per chunk, in input order
        chunks = _chunks([len(s) for _, s in items], max_residues)
        # one page-locked buffer per job in flight, reused chunk after chunk (rows are written out in on_done, before the buffer's
        # next chunk is submitted): a device-to-host copy into pageable memory returns only once it has completed, so every
        # submit would wait for its own chunk's kernels and nothing would overlap
        import torch
        rows_max = max((hi - lo for lo, hi in chunks), default=0)
        ring = [torch.empty((rows_max, predictor.n_terms), dtype=torch.float32, pin_memory=True).numpy() for _ in range(2)]

        def write(k: int, rows: np.ndarray) -> None:
            lo, hi = chunks[k]
            for (query_id, _), vec in zip(items[lo:hi], rows):
                tsv_writer.writerow([query_id, net_type] + vec.tolist())
        stream_chunks(lambda c, rows: predictor.submit_sequences([s for _, s in items[c[0]:c[1]]], out=rows),
                      ((c, c[1] - c[0]) for c in chunks), ring, depth=2, on_done=write)
        return
    if net_type != "gcn":
        raise ValueError(f"run_prediction_loop: unknown net_type {net_type!r}")
    lengths = [len(a.query_sequence) for a, _ in items]
    for lo, hi in _chunks(lengths, max_residues):
        seqs = [a.query_sequence for a, _ in items[lo:hi]]
        maps = [pack_bits(np.asarray(c)) for _, c in items[lo:hi]]
        scores = predictor.forward_batch(seqs, maps)
        for (aln, _), vec in zip(items[lo:hi], scores):
            tsv_writer.writerow([aln.query_name, net_type] + vec.tolist())


def predict_structures(predictors: Dict[str, Predictor], alignments: Sequence, threshold: float = 6,
                       generated_contacts: int = 2, max_residues: int = DEFAULT_MAX_RESIDUES,
                       writers: Optional[Dict[str, "csv.writer"]] = None):
    """Contact-map build + alignment transfer + GCN forward of every mode in `predictors` (`{"mf": Predictor, ...}`,
    all on one context) for all alignments that carry coordinates.

    Returns `(scores, kept, skipped)`: `scores[mode]` is float32 `[len(kept), C_mode]`, `kept` / `skipped` index
    `alignments` (skipped = no structure).  With `writers`, rows `[query_name, "gcn"] + scores` are also written
    per mode in input order, exactly what `pipeline.py:318-319` writes."""
    if not predictors:
        raise ValueError("predict_structures: no predictors")
    kept = [i for i, a in enumerate(alignments) if getattr(a, "coords", None) is not None]
    skipped = [i for i, a in enumerate(alignments) if getattr(a, "coords", None) is None]
    first = next(iter(predictors.values()))
    out = {mode: np.empty((len(kept), p.n_terms), np.float32) for mode, p in predictors.items()}
    lengths = [len(alignments[i].query_sequence) for i in kept]
    for lo, hi in _chunks(lengths, max_residues):
        part = [alignments[i] for i in kept[lo:hi]]
        batch = first.upload([a.query_sequence for a in part], [a.gapped_sequence for a in part],
                             [a.gapped_target for a in part], [np.ascontiguousarray(a.coords, np.float32) for a in part])
        try:
            for mode, pred in predictors.items():
                pred.run(batch, threshold, generated_contacts, share=True)   # maps and LM output come from the first head
                pred.fetch_scores(batch, out[mode][lo:hi])
        finally:
            batch.close()
        if writers:
            for mode, w in writers.items():
                for a, vec in zip(part, out[mode][lo:hi]):
                    w.writerow([a.query_name, "gcn"] + vec.tolist())
    return out, kept, skipped


def predict_pairs(predictors: Dict[str, Predictor], query_ids: Sequence[str], queries: Sequence[str], target_ids: Sequence[str],
                  targets: Sequence[str], coords: Sequence[np.ndarray], scoring_matrix="VTML80", gap_open: int = 10, gap_extend: int = 1,
                  threshold: float = 6, generated_contacts: int = 2, max_residues: int = DEFAULT_MAX_RESIDUES,
                  writers: Optional[Dict[str, "csv.writer"]] = None):
    """`predict_structures` from (query, best-hit target, target coordinates) pairs: `align_mmseqs_results` +
    `build_align_contact_map` + `forward_pass` of every mode in `predictors` (all on one context).  Per chunk the pairs are
    uploaded and aligned once (`Predictor.upload_pairs`), then every head runs on the batch with `share=True`.

    Returns `(scores, stats)`: `scores[mode]` is float32 `[n, C_mode]` in input order; `stats` holds per pair the `target_id`,
    the int32 `nw_score`, `aln_len` and `n_match` arrays and `identity` = n_match / aln_len (PyOpal's `identity()`).  With
    `writers`, rows `[query_id, "gcn"] + scores` are written per mode in input order, as `pipeline.py:318-319` writes them."""
    if not predictors:
        raise ValueError("predict_pairs: no predictors")
    n = len(queries)
    if not len(query_ids) == len(target_ids) == len(targets) == len(coords) == n:
        raise ValueError("predict_pairs: query_ids, queries, target_ids, targets and coords must have the same length")
    first = next(iter(predictors.values()))
    out = {mode: np.empty((n, p.n_terms), np.float32) for mode, p in predictors.items()}
    stats = {k: np.empty(n, np.int32) for k in ("nw_score", "aln_len", "n_match")}
    for lo, hi in _chunks([len(q) for q in queries], max_residues):
        batch = first.upload_pairs(queries[lo:hi], targets[lo:hi], coords[lo:hi], scoring_matrix, gap_open, gap_extend)
        try:
            for mode, pred in predictors.items():
                pred.run(batch, threshold, generated_contacts, share=True)   # maps and LM output come from the first head
                pred.fetch_scores(batch, out[mode][lo:hi])
            stats["nw_score"][lo:hi], stats["aln_len"][lo:hi], stats["n_match"][lo:hi] = batch.alignment()
        finally:
            batch.close()
        if writers:
            for mode, w in writers.items():
                for qid, vec in zip(query_ids[lo:hi], out[mode][lo:hi]):
                    w.writerow([qid, "gcn"] + vec.tolist())
    stats["identity"] = np.where(stats["aln_len"] > 0, stats["n_match"] / np.maximum(stats["aln_len"], 1), 0.0)
    stats["target_id"] = list(target_ids)
    return out, stats
