"""GPU tests of the asynchronous form of the sequence-only DeepCNN branch: `Predictor.submit_sequences` (C: mdf_cnn_submit_ragged
through the Python-list collector) against the synchronous `forward_sequences`, two jobs in flight, CNN and GCN jobs sharing the
context's two job slots, error reporting, the streamed prediction loop and the sharded run through `stream_chunks` + `ScoreBoard`.

The job runs the same kernels as `forward_sequences` on the same inputs and the max-pool does not depend on the order of the
residue tiles, so the two forms are compared for exact equality.  Wherever jobs are meant to be in flight together their scores go
to page-locked memory: a device-to-host copy into pageable memory returns only once it has completed, so a submit with a pageable
`out` would return after its own job had finished on the device."""
import csv
import gc
import os
import subprocess
import sys

import numpy as np
import pytest

import spec
from conftest import golden_workload
from metagenomic_deepfri_b200 import _lib, distributed, pipeline, predict, synth

pytestmark = pytest.mark.gpu
TOL = 1e-3
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def cnn(cnn_model_dir):
    preds = {tag: predict.Predictor(path) for tag, path in cnn_model_dir.items()}
    yield preds
    for p in preds.values():
        p.close()


def configs4_sequences(n, seed):
    """n sequences with the metagenomic length distribution of BASELINE configs[4] (L ~ LogNormal(250, 0.6) in [50, 1000])."""
    rng = np.random.default_rng(seed)
    lengths = np.clip(np.exp(rng.normal(np.log(250.0), 0.6, size=n)), 50, 1000).astype(np.int64)
    return synth.random_sequences(rng, lengths)


def pinned(n, c):
    import torch
    return torch.empty((n, c), dtype=torch.float32, pin_memory=True).numpy()


def alphabet_sequences(lengths, seed):
    rng = np.random.default_rng(seed)
    letters = np.array(list(spec.CNN_ALPHABET))
    return ["".join(rng.choice(letters, int(L))) for L in lengths]


@pytest.mark.parametrize("tag", list(spec.CNN_CASES))
def test_job_equals_synchronous_form_and_golden(cnn, cnn_golden, tag):
    pred = cnn[tag]
    seqs = spec.cnn_sequences(tag)
    got = pred.submit_sequences(seqs).wait()
    assert got.dtype == np.float32 and got.shape == (len(seqs), pred.n_terms)
    assert np.array_equal(got, pred.forward_sequences(seqs))
    assert np.abs(got - cnn_golden[f"{tag}_scores"]).max() <= TOL


def test_job_equals_synchronous_form_configs4_batch(cnn):
    pred = cnn["cnn_mf"]
    seqs = configs4_sequences(2048, 77)
    assert np.array_equal(pred.submit_sequences(seqs).wait(), pred.forward_sequences(seqs))


def test_two_jobs_in_flight(cnn):
    pred = cnn["cnn_small"]
    a = alphabet_sequences([1, 127, 128, 129, 513, 40, 700, 2], 3)
    b = alphabet_sequences([513, 129, 1, 128, 127] + list(np.random.default_rng(4).integers(1, 900, 3000)), 5)
    want_a, want_b = pred.forward_sequences(a), pred.forward_sequences(b)
    ja = pred.submit_sequences(a, out=pinned(len(a), pred.n_terms))
    jb = pred.submit_sequences(b, out=pinned(len(b), pred.n_terms))
    with pytest.raises(ValueError, match="both job slots"):
        pred.submit_sequences(["ACDE"])
    assert np.array_equal(jb.wait(), want_b)       # waited out of submission order
    assert np.array_equal(ja.wait(), want_a)
    assert ja.wait() is ja.wait()                  # a second wait returns the same matrix


def test_cnn_and_gcn_jobs_share_the_slots(cnn, model_dir):
    pred = cnn["cnn_small"]
    gcn = predict.Predictor(model_dir["tc_small"])
    try:
        assert gcn._ctx is pred._ctx                   # one context, one pair of job slots
        wl = golden_workload("tc_small")
        want_gcn = gcn.forward_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, 10.0, 2)
        seqs = configs4_sequences(3000, 8)
        want_cnn = pred.forward_sequences(seqs)
        for order in ("cnn_first", "gcn_first"):
            jobs = {}
            for kind in (("cnn", "gcn") if order == "cnn_first" else ("gcn", "cnn")):
                jobs[kind] = pred.submit_sequences(seqs, out=pinned(len(seqs), pred.n_terms)) if kind == "cnn" else \
                    gcn.submit_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, 10.0, 2,
                                          out=pinned(len(wl.query_seqs), gcn.n_terms))
            with pytest.raises(ValueError, match="both job slots"):
                pred.submit_sequences(seqs[:3])
            assert np.array_equal(jobs["cnn"].wait(), want_cnn)
            assert np.abs(jobs["gcn"].wait() - want_gcn).max() < 1e-5
    finally:
        gcn.close()


def test_caller_buffers_may_be_released(cnn):
    """The strings may go as soon as the submit returns.  Through the collector directly, so that nothing but the library could
    still refer to them (a PathJob keeps its list to name a bad residue); a 2,048-sequence job on the full-size model with its
    scores going to page-locked memory is still on the device when the list is dropped and its memory reused."""
    import ctypes as C
    pred = cnn["cnn_mf"]
    seqs = configs4_sequences(2048, 17)
    lengths = [len(s) for s in seqs]
    want = pred.forward_sequences(seqs)
    del seqs
    out = pinned(len(lengths), pred.n_terms)
    seqs = configs4_sequences(2048, 17)                 # fresh str objects, referenced by this list only
    rc, job = _lib.pyhost().submit_sequences(_lib.fn_addr("mdf_cnn_submit_ragged"), pred._handle.value, seqs, out.ctypes.data)
    _lib.check(rc)
    del seqs
    gc.collect()
    filler = ["W" * L for L in lengths]                 # fresh strings of the same sizes, likely in the freed memory
    _lib.check(_lib.lib().mdf_path_wait(C.c_void_p(job)))
    assert np.array_equal(out, want)
    del filler


def test_errors(cnn, model_dir):
    pred = cnn["cnn_small"]
    with pytest.raises(ValueError, match="Invalid character in sequence: J"):
        pred.submit_sequences(["ACDE", "ACJE"]).wait()
    with pytest.raises(ValueError, match="sequence 1 is empty"):
        pred.submit_sequences(["ACD", ""])
    with pytest.raises(UnicodeEncodeError):
        pred.submit_sequences(["ACD", "ACé"])
    gcn = predict.Predictor(model_dir["small"])
    try:
        with pytest.raises(ValueError):
            gcn.submit_sequences(["ACDE"])
    finally:
        gcn.close()
    for bad in (np.empty((2, pred.n_terms), np.float64), np.empty((3, pred.n_terms), np.float32),
                np.empty((pred.n_terms, 2), np.float32).T):
        with pytest.raises(ValueError, match="out must be"):
            pred.submit_sequences(["ACD", "EF"], out=bad)
    empty = pred.submit_sequences([]).wait()
    assert empty.shape == (0, pred.n_terms) and empty.dtype == np.float32
    # a failed job leaves no error behind: the next jobs on both slots are correct
    seqs = alphabet_sequences([300, 1, 129], 11)
    want = pred.forward_sequences(seqs)
    with pytest.raises(ValueError, match="Invalid character"):
        pred.submit_sequences(seqs + ["AAJ"]).wait()
    for _ in range(2):
        j1, j2 = pred.submit_sequences(seqs), pred.submit_sequences(seqs[::-1])
        assert np.array_equal(j1.wait(), want) and np.array_equal(j2.wait(), want[::-1])


def test_prediction_loop_streams_chunks(cnn, tmp_path):
    """run_prediction_loop(..., "cnn") with a residue limit that cuts the input into several chunks writes the rows of the
    reference's per-query loop (pipeline.py:313-319), bit for bit, in input order."""
    pred = cnn["cnn_small"]
    lengths = np.random.default_rng(12).integers(1, 400, 60)
    unaligned = {f"q{i}": s for i, s in enumerate(alphabet_sequences(lengths, 13))}
    max_residues = 2000
    assert len(pipeline._chunks(list(map(len, unaligned.values())), max_residues)) >= 3
    ref_rows = [[qid, "cnn"] + pred.forward_pass(seqres=s).tolist() for qid, s in unaligned.items()]
    out = tmp_path / "prediction_matrix_mf_cnn.tsv"
    with open(out, "w", newline="") as fh:
        pipeline.run_prediction_loop(pred, unaligned.items(), len(unaligned), "cnn", csv.writer(fh, delimiter="\t"),
                                     max_residues=max_residues)
    rows = list(csv.reader(open(out), delimiter="\t"))
    assert [r[:2] for r in rows] == [r[:2] for r in ref_rows]
    assert np.array_equal(np.array([r[2:] for r in rows], np.float32), np.array([r[2:] for r in ref_rows], np.float32))


def test_single_rank_stream_into_scoreboard(cnn):
    pred = cnn["cnn_small"]
    seqs = configs4_sequences(3000, 21)
    lengths = [len(s) for s in seqs]
    mine = distributed.shard_job(lengths, 1, max_proteins=700, max_residues=150_000, alpha=0.0)[0]
    assert len(mine) >= 3
    board = distributed.ScoreBoard(len(seqs), pred.n_terms)
    try:
        local = pinned(len(seqs), pred.n_terms)
        distributed.stream_chunks(lambda ch, rows: pred.submit_sequences([seqs[i] for i in ch], out=rows),
                                  ((c, len(c)) for c in mine), local, on_done=lambda k, rows: board.put(mine[k], rows))
        final = board.finish()
        assert np.array_equal(final, pred.forward_sequences(seqs))
        final = None
    finally:
        board.close()


def test_two_gpu_sharded_run(cnn_model_dir):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = os.path.join(ROOT, "tests", "_cnn_shard_worker.py")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29617")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29617", script, cnn_model_dir["cnn_small"]],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "CNN_SHARD_OK" in r.stdout
