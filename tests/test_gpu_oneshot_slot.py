"""GPU tests of the synchronous calls (`forward_pass`, `forward_batch`, `build_align_contact_maps`, `mdf_cmap_build_transfer`,
`forward_sequences`) while asynchronous jobs are in flight.  They run in the context's own synchronous job slot, which the ring of
`submit_*` never hands out: with both ring slots busy every one of them succeeds, returns what it returns with nothing in flight,
keeps its error texts, and leaves the jobs in flight intact.

Contact maps and DeepCNN scores are compared for exact equality.  GCN scores are compared to 1e-5: both GCN engines sum-pool with
float atomics, so their last bits may differ from run to run.  The jobs' scores go to page-locked memory, so that a submit returns
while its job is still on the device."""
import numpy as np
import pytest

import cmap_oracle as co
from conftest import Aln, golden_workload
from metagenomic_deepfri_b200 import _lib, batching, bio_utils, predict, synth

pytestmark = pytest.mark.gpu
GCN_TOL = 1e-5


def pinned(n, c):
    import torch
    return torch.empty((n, c), dtype=torch.float32, pin_memory=True).numpy()


@pytest.fixture(scope="module")
def preds(model_dir, cnn_model_dir):
    gcn, cnn = predict.Predictor(model_dir["tc_small"]), predict.Predictor(cnn_model_dir["cnn_small"])
    assert gcn._ctx is cnn._ctx                      # one context: one ring of two job slots and one synchronous slot
    yield gcn, cnn
    gcn.close()
    cnn.close()


@pytest.fixture(scope="module")
def wl():
    return golden_workload("tc_small")


@pytest.fixture(scope="module")
def seqs():
    rng = np.random.default_rng(31)
    return synth.random_sequences(rng, np.clip(np.exp(rng.normal(np.log(250.0), 0.6, size=3000)), 50, 1000).astype(np.int64))


class Ring:
    """Both ring slots busy: a structure job and a sequence job, submitted into page-locked outputs."""

    def __init__(self, gcn, cnn, wl, seqs):
        self.gcn_job = gcn.submit_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, 10.0, 2,
                                             out=pinned(len(wl.query_seqs), gcn.n_terms))
        self.cnn_job = cnn.submit_sequences(seqs, out=pinned(len(seqs), cnn.n_terms))

    def check(self, want_gcn, want_cnn):
        assert np.abs(self.gcn_job.wait() - want_gcn).max() < GCN_TOL
        assert np.array_equal(self.cnn_job.wait(), want_cnn)


def alone(gcn, cnn, wl, seqs):
    return (gcn.forward_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, 10.0, 2),
            cnn.forward_sequences(seqs))


def flat_cmap(wl, packed):
    """`mdf_cmap_build_transfer` on flat buffers; packed: canonical packed_off -> uint32 words, else dense int32 cells."""
    ps = batching.pack_structures(wl.gapped_query, wl.gapped_target, wl.coords)
    lens = np.diff(ps.seq_off)
    dense_off = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens * lens, out=dense_off[1:])
    buf = np.zeros(int(ps.packed_off[-1] if packed else dense_off[-1]), np.uint32 if packed else np.int32)
    _lib.check(_lib.lib().mdf_cmap_build_transfer(
        _lib.default_context().handle, ps.n, _lib.fp(ps.coords), _lib.lp(ps.coord_off), ps.q_aln, ps.t_aln, _lib.lp(ps.aln_off),
        _lib.lp(ps.seq_off), 100.0, 2, _lib.up(buf) if packed else None, _lib.lp(ps.packed_off) if packed else None,
        None if packed else _lib.ip(buf), None if packed else _lib.lp(dense_off)))
    return buf


def test_synchronous_calls_while_two_jobs_are_in_flight(preds, wl, seqs):
    gcn, cnn = preds
    alns = [Aln(q, t, c, i) for i, (q, t, c) in enumerate(zip(wl.gapped_query, wl.gapped_target, wl.coords))]
    packed = bio_utils.build_align_contact_maps(alns, 10.0, 2, packed=True)
    words = sum(m.size for m in packed)
    dense0 = co.build_align_contact_map(wl.gapped_query[0], wl.gapped_target[0], wl.coords[0], 10.0, 2).astype(np.int32)
    short = seqs[:200]

    def calls():
        arena = np.zeros(words, np.uint32)
        return {"forward_pass": gcn.forward_pass(wl.query_seqs[0], dense0),
                "forward_batch": gcn.forward_batch(wl.query_seqs, packed),
                "maps_into_out": [m.copy() for m in bio_utils.build_align_contact_maps(alns, 10.0, 2, packed=True, out=arena)],
                "maps_dense": bio_utils.build_align_contact_maps(alns, 10.0, 2),
                "flat_packed": flat_cmap(wl, True), "flat_dense": flat_cmap(wl, False),
                "forward_sequences": cnn.forward_sequences(short)}

    want = calls()
    want_gcn, want_cnn = alone(gcn, cnn, wl, seqs)
    ring = Ring(gcn, cnn, wl, seqs)
    with pytest.raises(ValueError, match="both job slots"):
        cnn.submit_sequences(short)
    got = calls()
    for k in ("forward_pass", "forward_batch"):
        assert np.abs(got[k] - want[k]).max() < GCN_TOL, k
    for k in ("maps_into_out", "maps_dense"):
        assert all(np.array_equal(a, b) for a, b in zip(got[k], want[k])), k
    for k in ("flat_packed", "flat_dense", "forward_sequences"):
        assert np.array_equal(got[k], want[k]), k
    ring.check(want_gcn, want_cnn)


def test_synchronous_call_between_two_submits(preds, wl, seqs):
    """submit A; forward_batch; submit B: the synchronous call takes no ring slot, so B is the second job in flight."""
    gcn, cnn = preds
    packed = bio_utils.build_align_contact_maps([Aln(q, t, c) for q, t, c in zip(wl.gapped_query, wl.gapped_target, wl.coords)],
                                                10.0, 2, packed=True)
    want_batch = gcn.forward_batch(wl.query_seqs, packed)
    want_gcn, want_cnn = alone(gcn, cnn, wl, seqs)
    a = gcn.submit_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, 10.0, 2,
                              out=pinned(len(wl.query_seqs), gcn.n_terms))
    assert np.abs(gcn.forward_batch(wl.query_seqs, packed) - want_batch).max() < GCN_TOL
    b = cnn.submit_sequences(seqs, out=pinned(len(seqs), cnn.n_terms))
    assert np.array_equal(b.wait(), want_cnn)
    assert np.abs(a.wait() - want_gcn).max() < GCN_TOL


def test_synchronous_errors_keep_their_texts_and_leave_the_jobs_intact(preds, wl, seqs):
    gcn, cnn = preds
    L = _lib.lib()
    want_gcn, want_cnn = alone(gcn, cnn, wl, seqs)
    good = np.eye(4, dtype=np.int32)
    want_pass = gcn.forward_pass("ACDE", good)
    ring = Ring(gcn, cnn, wl, seqs)
    y = np.empty(gcn.n_terms, np.float32)
    bad_map = good.copy()
    bad_map[1, 2] = 2
    with pytest.raises(ValueError, match="Invalid character in sequence: J"):
        gcn.forward_batch(["ACJE"], [np.zeros((4, 4), np.uint32)])
    # past the Python-side check: the device flags the residue, the library names the call
    seq_off = np.array([0, 4], np.int64)
    with pytest.raises(ValueError, match="^path: Invalid character in sequence"):
        _lib.check(L.mdf_gcn_forward_packed(gcn._handle, 1, b"ACJE", _lib.lp(seq_off), _lib.up(np.zeros(16, np.uint32)),
                                            _lib.lp(batching.packed_offsets(np.array([4]))), _lib.fp(y)))
    with pytest.raises(ValueError, match="^forward_pass: contact map holds values other than 0/1"):
        gcn.forward_pass("ACDE", bad_map)
    with pytest.raises(ValueError, match="^path: Invalid character in sequence"):    # both faults: the residue comes first
        _lib.check(L.mdf_gcn_forward_dense(gcn._handle, b"ACJE", 4, _lib.ip(bad_map), _lib.fp(y)))
    ps = batching.pack_structures(wl.gapped_query, wl.gapped_target, wl.coords)
    shifted = ps.packed_off.copy()
    shifted[1:] += 4
    buf = np.zeros(int(shifted[-1]), np.uint32)
    with pytest.raises(ValueError, match=r"packed_off\[1\] is not canonical"):
        _lib.check(L.mdf_cmap_build_transfer(_lib.default_context().handle, ps.n, _lib.fp(ps.coords), _lib.lp(ps.coord_off), ps.q_aln,
                                             ps.t_aln, _lib.lp(ps.aln_off), _lib.lp(ps.seq_off), 100.0, 2, _lib.up(buf),
                                             _lib.lp(shifted), None, None))
    with pytest.raises(ValueError, match="sequence 1 is empty"):
        cnn.forward_sequences(["ACD", ""])
    # no error is left behind for the next synchronous call, and the jobs return what they return alone
    assert np.abs(gcn.forward_pass("ACDE", good) - want_pass).max() < GCN_TOL
    ring.check(want_gcn, want_cnn)
