"""CPU tests of the float64 stage reference (`oracle/gcn_f64.py`) that tests/test_gpu_tc_shapes.py measures both engines
against: every stage it returns agrees with the fp32 ONNX interpreter's node of the same name on shapes of the tensor-core
shape matrix, and the batched LSTM, which steps all proteins in lockstep, gives each protein what it computes alone."""
import numpy as np
import pytest

import cmap_oracle as co
import gcn_f64
import gcn_oracle as go
import spec
from metagenomic_deepfri_b200 import synth

# shapes of spec.TC_SHAPES that together cover H = 192, gc (384, 128), four layers, Relu + bias and n_terms = 1
CASES = ["h192", "h256", "h320", "h64_relu_bias"]
LENGTHS = (1, 2, 17, 40, 33)


def _case(tag):
    kw, seed, _, _ = spec.TC_SHAPES[tag]
    cfg = synth.GCNConfig(**kw)
    return cfg, synth.make_weights(cfg, seed), seed


def _rel(got, want):
    """max |got - want| over the largest |want| (at least 1)."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape
    return float(np.abs(got - want).max() / max(1.0, np.abs(want).max()))


@pytest.mark.parametrize("tag", CASES)
def test_stages_match_onnx_oracle(tag, tmp_path):
    cfg, w, seed = _case(tag)
    path = str(tmp_path / f"{tag}.onnx")
    synth.write_gcn_model(path, cfg, seed=seed)
    oracle = go.OnnxOracle(path)
    wl, cms = spec.structure_batch(LENGTHS, seed)
    ref = gcn_f64.reference(w, cfg, wl.query_seqs, cms)
    act = cfg.gc_activation
    nodes = ["lm/LSTM1_out", "lm/LSTM2_bm", "activation/Relu"] + [f"GraphConv_{l}/{act}" for l in range(1, len(cfg.gc_dims) + 1)] + \
            ["norm/d", "SumPooling/Sum", "labels"]
    off = ref["off"]
    for p, (seq, cm) in enumerate(zip(wl.query_seqs, cms)):
        L = len(seq)
        outs = dict(zip(nodes, oracle.run(nodes, {"cmap": cm[None].astype(np.float32), "seq": co.seq2onehot(seq)[None]})))
        rows = slice(off[p], off[p + 1])
        assert _rel(outs["lm/LSTM1_out"].reshape(L, -1), ref["h1"][rows]) < 1e-5, (tag, p, "lstm1")
        assert _rel(outs["lm/LSTM2_bm"].reshape(L, -1), ref["h2"][rows]) < 1e-5, (tag, p, "lstm2")
        assert _rel(outs["activation/Relu"].reshape(L, -1), ref["x0"][rows]) < 1e-5, (tag, p, "x0")
        for l in range(len(cfg.gc_dims)):
            assert _rel(outs[f"GraphConv_{l + 1}/{act}"].reshape(L, -1), ref["gc"][l][rows]) < 1e-5, (tag, p, f"gc{l + 1}")
        assert _rel(outs["norm/d"].reshape(L), ref["d"][rows]) < 1e-6, (tag, p, "d")
        assert _rel(outs["SumPooling/Sum"].reshape(-1), ref["pooled"][p]) < 1e-5, (tag, p, "pooled")
        lab = outs["labels"].reshape(-1, 2)
        assert np.abs(lab[:, 0] - ref["scores"][p]).max() < 2e-6, (tag, p, "scores")
        e = np.exp(ref["logits"][p] - ref["logits"][p].max(1, keepdims=True))
        assert np.abs(lab - e / e.sum(1, keepdims=True)).max() < 2e-6, (tag, p, "labels")


@pytest.mark.parametrize("tag", ["h192", "h64_relu_bias"])
def test_batched_lstm_equals_per_protein(tag):
    """Stepping proteins of 1 ... 300 residues in lockstep leaks nothing across proteins: each one gets, to float64
    rounding, every stage it gets alone, and the scores of the one-protein restatement `deepfri_numpy`."""
    cfg, w, seed = _case(tag)
    lengths = [1, 300, 2, 64, 65, 17, 299, 1, 128, 129, 250]
    wl, cms = spec.structure_batch(lengths, seed + 1)
    batch = gcn_f64.reference(w, cfg, wl.query_seqs, cms)
    off = batch["off"]
    for p, (seq, cm) in enumerate(zip(wl.query_seqs, cms)):
        one = gcn_f64.reference(w, cfg, [seq], [cm])
        rows = slice(off[p], off[p + 1])
        for k in ("h1", "h2", "x0", "d"):
            assert np.abs(batch[k][rows] - one[k]).max() <= 1e-12, (p, k)
        for l in range(len(cfg.gc_dims)):
            assert np.abs(batch["gc"][l][rows] - one["gc"][l]).max() <= 1e-12, (p, l)
        assert np.abs(batch["pooled"][p] - one["pooled"][0]).max() <= 1e-10 * max(1.0, np.abs(one["pooled"]).max())
        assert np.abs(batch["scores"][p] - one["scores"][0]).max() <= 1e-12
        assert np.abs(batch["scores"][p] - gcn_f64.deepfri_numpy(w, cfg, seq, cm)).max() <= 1e-12
