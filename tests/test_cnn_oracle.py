"""CPU tests of the sequence-only DeepCNN branch (predict.pyx:91-95): the ONNX interpreter's Conv / BatchNormalization /
ReduceMax against an independent float64 restatement of upstream DeepFRI's DeepCNN equations, the graph recogniser, and the
frozen golden vectors."""
import os

import numpy as np
import pytest

import gcn_oracle as go
from cnn_f64 import deepcnn_f64
from metagenomic_deepfri_b200 import onnx_lite as ox
from metagenomic_deepfri_b200 import synth
from metagenomic_deepfri_b200._lib import UnsupportedModelError
from conftest import recognise
import spec

ALPHABET = "-DGULNTKHYWCPVSOIEFXQABZRM"


@pytest.mark.parametrize("tag", ["cnn_small"])
def test_oracle_matches_independent_restatement(tag, tmp_path):
    kw, seed, n, lo, hi = spec.CNN_CASES[tag]
    cfg = synth.CNNConfig(**kw)
    w = synth.make_cnn_weights(cfg, seed)
    path = str(tmp_path / "cnn.onnx")
    ox.save(synth.build_cnn_model(cfg, w), path)
    orc = go.Predictor(path)
    assert orc.input_names == ["seq"]
    rng = np.random.default_rng(5)
    for L in (1, 2, 7, 33, 150):
        seq = "".join(rng.choice(list(ALPHABET), L))
        got = orc.forward_pass(seq)
        want = deepcnn_f64(w, cfg, seq)
        assert got.dtype == np.float32 and got.shape == (cfg.n_terms,)
        assert np.abs(got - want).max() < 2e-6


def test_cnn_plan_reads_graph():
    cfg = synth.CNNConfig(filter_lens=(5, 8, 16), num_filters=(128, 256, 128), n_terms=17)
    w = synth.make_cnn_weights(cfg, 3)
    plan = recognise(synth.build_cnn_model(cfg, w))
    assert plan.kind == "cnn" and plan.input_names == ["seq"] and plan.n_terms == 17
    assert plan.conv_filters == [128, 256, 128] and plan.conv_width == [5, 8, 16]
    assert plan.conv_pad_left == [2, 3, 7]
    for l in (1, 2, 3):
        assert np.array_equal(plan.tensor(f"conv{l}_W"), w[f"conv1d_{l}_W"].reshape(-1))      # [F, 26, 1, w] == [F, 26, w] flat
    s = w["bn_gamma"].astype(np.float64) / np.sqrt(w["bn_var"].astype(np.float64) + cfg.bn_epsilon)
    b = np.concatenate([w[f"conv1d_{l}_b"] for l in (1, 2, 3)])
    assert np.allclose(plan.tensor("scale"), s, rtol=1e-6)
    assert np.allclose(plan.tensor("shift"), (b - w["bn_mean"]) * s + w["bn_beta"], rtol=1e-5, atol=1e-6)
    assert np.array_equal(plan.tensor("out_W"), w["labels_W"].reshape(-1)) and np.array_equal(plan.tensor("out_b"), w["labels_b"])


def test_cnn_plan_rejects_foreign_graphs():
    cfg = synth.CNNConfig(filter_lens=(5, 8), num_filters=(128, 128), n_terms=9)
    m = synth.build_cnn_model(cfg)
    g = m.graph
    gcn = synth.build_gcn_model(synth.GCNConfig(**spec.SMALL)).graph   # a GCN body behind a single input is not a DeepCNN
    with pytest.raises(UnsupportedModelError):
        recognise(ox.Model(ox.Graph(nodes=gcn.nodes, initializers=gcn.initializers, inputs=[gcn.inputs[1]], outputs=gcn.outputs)))
    nodes = [n for n in g.nodes if n.op_type != "Relu"]
    with pytest.raises(UnsupportedModelError):
        recognise(ox.Model(ox.Graph(nodes=nodes, initializers=g.initializers, inputs=g.inputs, outputs=g.outputs)))
    import copy
    g2 = copy.deepcopy(g)
    for n in g2.nodes:
        if n.op_type == "Conv":
            n.attrs["pads"] = [0, 0, 0, 0]                         # 'valid' padding changes the output length
            break
    with pytest.raises(UnsupportedModelError, match="same"):
        recognise(ox.Model(g2))


def test_cnn_golden_matches_oracle(cnn_golden, cnn_model_dir):
    """The committed golden scores are what the oracle computes today (guards the oracle against drift)."""
    for tag, (kw, seed, n, lo, hi) in spec.CNN_CASES.items():
        seqs = spec.cnn_sequences(tag)
        orc = go.Predictor(cnn_model_dir[tag])
        want = cnn_golden[f"{tag}_scores"]
        assert want.shape == (len(seqs), kw["n_terms"])
        for i in spec.CNN_GOLDEN_CHECK[tag]:
            assert np.abs(orc.forward_pass(seqs[i]) - want[i]).max() < 1e-6


def test_cnn_plan_accepts_equivalent_lowerings(tmp_path):
    """tf2onnx versions lower the same Keras layers differently: `auto_pad=SAME_UPPER` instead of explicit pads, rank-3 Conv
    weights, a Gemm instead of MatMul + Add, GlobalMaxPool instead of ReduceMax.  The recogniser must read the same plan and
    the oracle must give the same scores for all of them."""
    import copy
    cfg = synth.CNNConfig(filter_lens=(4, 9), num_filters=(128, 128), n_terms=7, logit_scale=0.5)
    base = synth.build_cnn_model(cfg, seed=8)
    ref_plan = recognise(base)

    def variant(edit):
        m = ox.loads(ox.dumps(base))
        edit(m.graph)
        return m

    def auto_pad(g):
        for n in g.nodes:
            if n.op_type == "Conv":
                n.attrs.pop("pads")
                n.attrs["auto_pad"] = "SAME_UPPER"

    def gemm_head(g):
        mm = next(n for n in g.nodes if n.op_type == "MatMul")
        add = next(n for n in g.nodes if n.op_type == "Add" and mm.outputs[0] in n.inputs)
        bias = [i for i in add.inputs if i != mm.outputs[0]][0]
        g.nodes[g.nodes.index(mm)] = ox.Node("Gemm", [mm.inputs[0], mm.inputs[1], bias], [add.outputs[0]], name="Gemm__head", attrs={})
        g.nodes.remove(add)

    variants = {"auto_pad": variant(auto_pad), "gemm": variant(gemm_head)}
    seqs = ["ACDEFGHIKLMNPQRSTVWY", "MK", "W" * 40 + "ACD"]
    p0 = str(tmp_path / "base.onnx")
    ox.save(base, p0)
    want = [go.Predictor(p0).forward_pass(s) for s in seqs]
    for tag, m in variants.items():
        plan = recognise(m)
        assert plan.conv_pad_left == ref_plan.conv_pad_left and plan.n_terms == ref_plan.n_terms, tag
        for role in ("scale", "shift", "out_W", "out_b"):
            assert np.array_equal(plan.tensor(role), ref_plan.tensor(role)), (tag, role)
        pth = str(tmp_path / f"{tag}.onnx")
        ox.save(m, pth)
        orc = go.Predictor(pth)
        for s, w in zip(seqs, want):
            assert np.abs(orc.forward_pass(s) - w).max() < 1e-6, tag
