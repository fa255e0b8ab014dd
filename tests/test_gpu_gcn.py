"""GPU parity tests of the GCN half and of the whole path, through the C ABI, against the oracle.

Tolerance (BASELINE.json north_star): GO-term scores <= 1e-3 absolute, and identical calls at the
reference's reporting threshold (score >= 0.1, pipeline.py:701) outside a guard band of that
tolerance around 0.1 - a score the oracle itself puts within 1e-3 of the threshold cannot be pinned
by any arithmetic that is not bit-identical."""
import numpy as np
import pytest

import cmap_oracle as co
import gcn_oracle as go
import spec
from conftest import golden_workload
from metagenomic_deepfri_b200 import batching, predict, synth

pytestmark = pytest.mark.gpu
TOL = 1e-3
TOL_SIMT = 2e-5          # the exact-fp32 engine must sit on top of the oracle


def assert_scores(got, want, tol=TOL):
    assert got.shape == want.shape and got.dtype == np.float32
    err = np.abs(got - want).max() if got.size else 0.0
    assert err <= tol, f"max |score - oracle| = {err:.3e} > {tol}"
    clear = np.abs(want - 0.1) > tol
    assert np.array_equal((got >= 0.1)[clear], (want >= 0.1)[clear]), "GO calls differ outside the guard band"


def oracle_maps(wl):
    return [co.build_align_contact_map(wl.gapped_query[i], wl.gapped_target[i], wl.coords[i], wl.threshold,
                                       wl.generated_contacts) for i in range(len(wl))]


@pytest.fixture(scope="module")
def engines(model_dir):
    preds = {tag: predict.Predictor(p) for tag, p in model_dir.items()}
    yield preds
    for p in preds.values():
        p.close()


@pytest.mark.parametrize("tag", list(spec.GCN_CASES))
@pytest.mark.parametrize("engine", ["simt", "tc"])
def test_golden_scores(tag, engine, engines, gcn_golden):
    pred = engines[tag]
    try:
        pred.set_engine(engine)
    except ValueError:
        pytest.skip(f"{engine} engine unavailable for this model shape")
    wl = golden_workload(tag)
    cms = oracle_maps(wl)
    want = gcn_golden[tag + "_scores"]
    tol = TOL_SIMT if engine == "simt" else TOL
    for i in range(len(wl)):
        y = pred.forward_pass(wl.query_seqs[i], cms[i])             # predict.pyx:75-102 contract
        assert y.shape == (pred.n_terms,)
        assert_scores(y, want[i], tol)
    assert_scores(pred.forward_batch(wl.query_seqs, [batching.pack_bits(c) for c in cms]), want, tol)
    got = pred.forward_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, wl.threshold,
                                  wl.generated_contacts)
    assert_scores(got, want, tol)


@pytest.mark.parametrize("engine", ["simt", "tc"])
def test_path_against_oracle_config0_sample(engine, engines, model_dir):
    """A seeded sample of BASELINE config 0 (L 100-500, 10 A, MF head) end to end."""
    pred = engines["mf"]
    try:
        pred.set_engine(engine)
    except ValueError:
        pytest.skip("engine unavailable")
    oracle = go.Predictor(model_dir["mf"])
    wl = synth.config_workload(0, 0.024)           # 24 proteins
    want = np.stack([oracle.forward_pass(s, c) for s, c in zip(wl.query_seqs, oracle_maps(wl))])
    got = pred.forward_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, wl.threshold,
                                  wl.generated_contacts)
    assert_scores(got, want, TOL_SIMT if engine == "simt" else TOL)
    # stage taps against the oracle's node outputs (fp32 taps of both engines)
    b = pred.upload(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords)
    pred.run(b, wl.threshold, wl.generated_contacts)
    assert_scores(pred.fetch_scores(b), want, TOL_SIMT if engine == "simt" else TOL)
    packed = pred.fetch(b, "packed")
    for i, cm in enumerate(oracle_maps(wl)):
        L = cm.shape[0]
        rows = packed[b.packed_off[i]:b.packed_off[i + 1]].reshape(L, -1)
        assert np.array_equal(batching.unpack_bits(rows, L), cm)     # bit-exact inside the fused path too
    if engine == "simt":
        sess = oracle.session
        taps = {"lstm1": "lm/LSTM1_out", "lstm2": "lm/LSTM2_bm", "x0": "activation/Relu", "gc_last": "GraphConv_3/Elu"}
        cm0 = oracle_maps(wl)[0]
        outs = sess.run(list(taps.values()) + ["norm/d", "SumPooling/Sum"],
                        {"cmap": cm0[None].astype(np.float32), "seq": co.seq2onehot(wl.query_seqs[0])[None]})
        L0 = len(wl.query_seqs[0])
        for (k, _), o in zip(taps.items(), outs):
            g = pred.fetch(b, k)[:L0]
            assert np.abs(g - np.asarray(o).reshape(g.shape)).max() < 1e-4, k
        assert np.array_equal(pred.fetch(b, "deg")[:L0], outs[-2].reshape(-1))
        assert np.allclose(pred.fetch(b, "pooled")[0], outs[-1].reshape(-1), rtol=1e-5, atol=1e-3)
    b.close()


@pytest.mark.parametrize("layers", [1, 3])
def test_lstm_depth_other_than_two_runs_on_simt(layers, tmp_path):
    """The tensor-core engine computes the two-layer LSTM-LM that DeepFRI ships.  A model of another depth gets the exact-fp32
    engine, which runs any depth, and cannot be switched to the tensor-core one."""
    kw, seed, n, lo, hi = spec.GCN_CASES["tc_small"]
    path = str(tmp_path / f"lstm{layers}.onnx")
    synth.write_gcn_model(path, synth.GCNConfig(lstm_layers=layers, **kw), seed=seed)
    pred = predict.Predictor(path)
    try:
        assert pred.engine == "simt"
        with pytest.raises(ValueError, match="unavailable"):
            pred.set_engine("tc")
        wl = golden_workload("tc_small")
        oracle = go.Predictor(path)
        want = np.stack([oracle.forward_pass(s, c) for s, c in zip(wl.query_seqs, oracle_maps(wl))])
        got = pred.forward_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, wl.threshold,
                                      wl.generated_contacts)
        assert_scores(got, want, TOL_SIMT)
    finally:
        pred.close()


def test_batch_invariance_and_order(engines):
    """Scores of a protein do not depend on what else is in the batch or on its position."""
    pred = engines["small"]
    pred.set_engine("simt")
    wl = synth.make_workload(40, 1, 300, seed=77, threshold=10.0)
    full = pred.forward_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, 10.0, 2)
    perm = np.random.default_rng(1).permutation(len(wl))
    sub = lambda xs: [xs[i] for i in perm]
    shuffled = pred.forward_structures(sub(wl.query_seqs), sub(wl.gapped_query), sub(wl.gapped_target), sub(wl.coords), 10.0, 2)
    assert np.abs(shuffled - full[perm]).max() < 1e-5
    one = pred.forward_structures(wl.query_seqs[:1], wl.gapped_query[:1], wl.gapped_target[:1], wl.coords[:1], 10.0, 2)
    assert np.abs(one[0] - full[0]).max() < 1e-5
    assert pred.forward_structures([], [], [], [], 10.0, 2).shape == (0, pred.n_terms)


def test_forward_pass_contract_and_errors(engines):
    pred = engines["small"]
    assert pred.model_path.endswith("small.onnx") and pred.threads == 1 and pred.input_names == ["cmap", "seq"]
    assert [a.name for a in pred.session.get_inputs()] == pred.input_names
    cm = np.eye(4, dtype=np.int32)
    y = pred.forward_pass("ACDE", cm)
    assert y.dtype == np.float32 and y.shape == (24,) and np.all((y >= 0) & (y <= 1))
    assert np.array_equal(y, pred.forward_pass("ACDE", cm.astype(np.float32)))      # reference casts with astype
    assert np.array_equal(y, pred.forward_pass("ACDE", np.zeros((4, 4), np.int32)))  # diagonal is forced to 1
    with pytest.raises(ValueError, match="Invalid character in sequence: J"):
        pred.forward_pass("ACJE", cm)
    with pytest.raises(ValueError):
        pred.forward_pass("ACD", cm)                                                # shape mismatch
    with pytest.raises(ValueError):
        pred.forward_pass("ACDE", 3 * cm)
    with pytest.raises(ValueError, match="DeepCNN"):
        pred.forward_pass("ACDE")                                                   # a GCN head has no sequence-only branch
    with pytest.raises(ValueError):
        pred.forward_structures(["ACDE"], ["ACD-"], ["ACDE"], [np.zeros((4, 3), np.float32)])
    with pytest.raises(FileNotFoundError):
        predict.Predictor("/nonexistent/model.onnx")


def test_pipeline_loop_drop_in(engines, tmp_path):
    """The reference's prediction loop (pipeline.py:292-319) runs unchanged over the drop-in
    Predictor: same call, same row format as tests/test_pipeline_regression.py asserts."""
    import csv
    from conftest import Aln
    from metagenomic_deepfri_b200 import bio_utils
    pred = engines["small"]
    wl = synth.make_workload(5, 10, 60, seed=2, threshold=6.0)
    alns = [Aln(wl.gapped_query[i], wl.gapped_target[i], wl.coords[i], i) for i in range(len(wl))]
    pairs = [bio_utils.build_align_contact_map(a, threshold=6, generated_contacts=2) for a in alns]   # pipeline.py:476-481
    pairs = sorted([p for p in pairs if p[1] is not None], key=lambda x: len(x[0].query_sequence))    # :485,:529
    out = tmp_path / "prediction_matrix_mf.tsv"
    with open(out, "w", newline="") as fh:
        w = csv.writer(fh, delimiter="\t")
        for aln, cmap in pairs:                                                                         # :301-319
            vec = pred.forward_pass(seqres=aln.query_sequence, cmap=cmap)
            w.writerow([aln.query_name, "gcn"] + vec.tolist())
    rows = list(csv.reader(open(out), delimiter="\t"))
    assert len(rows) == 5 and all(r[1] == "gcn" and len(r) == 2 + pred.n_terms for r in rows)
