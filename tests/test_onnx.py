"""CPU tests: ONNX wire format, graph recognition by the library's own loader (`csrc/onnx_load.cu` through
`mdf_onnx_inspect` / `mdf_onnx_tensor`: host-only entry points, no GPU needed), and the GCN oracle against an independent
NumPy restatement of upstream DeepFRI's layer equations (SURVEY.md §3.3, `oracle/gcn_f64.py`)."""
import numpy as np
import pytest

import cmap_oracle as co
import gcn_oracle as go
from gcn_f64 import deepfri_numpy
from conftest import golden_workload, recognise
from metagenomic_deepfri_b200 import onnx_lite as ox
from metagenomic_deepfri_b200 import synth
from metagenomic_deepfri_b200._lib import UnsupportedModelError
import spec


def test_wire_roundtrip():
    m = synth.build_gcn_model(synth.GCNConfig(**spec.SMALL), seed=3)
    m2 = ox.loads(ox.dumps(m))
    assert [(n.op_type, n.inputs, n.outputs, n.attrs) for n in m2.graph.nodes] == \
           [(n.op_type, n.inputs, n.outputs, n.attrs) for n in m.graph.nodes]
    for k, v in m.graph.initializers.items():
        assert v.dtype == m2.graph.initializers[k].dtype and np.array_equal(v, m2.graph.initializers[k])
    assert [v.name for v in m2.graph.inputs] == ["cmap", "seq"] and m2.opset == 15
    assert m2.graph.inputs[1].shape[-1] == 26


def test_load_errors(tmp_path):
    with pytest.raises(FileNotFoundError):
        ox.load(str(tmp_path / "missing.onnx"))
    bad = tmp_path / "bad.onnx"
    bad.write_bytes(b"\xff\xff\xff\xffnot a protobuf")
    with pytest.raises(RuntimeError):
        ox.load(str(bad))


@pytest.mark.parametrize("style", ["compact", "tf2onnx"])
@pytest.mark.parametrize("kw", [dict(), dict(gc_activation="Relu", gc_bias=True, n_terms=320),
                                dict(lstm_hidden=256, gc_dims=(256, 128), fc_dim=512, n_terms=40)])
def test_plan_reads_hyperparameters_from_graph(kw, style):
    cfg = synth.GCNConfig(**kw)
    w = synth.make_weights(cfg, seed=11)
    plan = recognise(synth.build_gcn_model(cfg, w, style=style))
    assert plan.kind == "gcn" and plan.input_names == ["cmap", "seq"]
    assert plan.lstm_hidden == cfg.lstm_hidden and plan.lm_dim == cfg.lm_dim and plan.n_terms == cfg.n_terms
    assert plan.gc_dims == list(cfg.gc_dims) and plan.fc_dim == cfg.fc_dim and plan.n_lstm == 2
    assert plan.gc_activation == {"Relu": 1, "Elu": 2}[cfg.gc_activation]
    assert all((f"gc{l + 1}_b" in plan.roles) == cfg.gc_bias for l in range(len(cfg.gc_dims)))
    assert np.float32(plan.eps) == np.float32(cfg.eps)
    # every weight is found by its role in the dataflow (names below are what synth happened to call them)
    assert plan.roles["lm_W"] == "LM_embedding_W" and plan.roles["aa_W"] == "AA_embedding_W" and plan.roles["out_W"] == "labels_W"
    for role, name in (("lm_W", "LM_embedding_W"), ("aa_W", "AA_embedding_W"), ("fc_W", "dense_W"), ("out_W", "labels_W"),
                       ("lstm2_R", "lstm2_R"), ("lstm1_W", "lstm1_W"), ("lstm2_B", "lstm2_B"), ("gc2_W", "GraphConv_2_W"),
                       ("fc_b", "dense_b"), ("lm_b", "LM_embedding_b")):
        assert np.array_equal(plan.tensor(role), w[name].reshape(-1)), role
    if cfg.gc_bias:
        assert np.array_equal(plan.tensor("gc1_b"), w["GraphConv_1_b"])


def test_plan_rejects_foreign_graphs():
    m = synth.build_gcn_model(synth.GCNConfig(**spec.SMALL))
    g = m.graph
    swapped = ox.Model(ox.Graph(nodes=g.nodes, initializers=g.initializers, inputs=g.inputs[::-1], outputs=g.outputs))
    with pytest.raises(UnsupportedModelError, match="ordered"):
        recognise(swapped)
    no_sm = ox.Model(ox.Graph(nodes=g.nodes[:-1], initializers=g.initializers, inputs=g.inputs, outputs=g.outputs))
    with pytest.raises(UnsupportedModelError, match="Softmax"):
        recognise(no_sm)
    three = ox.Model(ox.Graph(nodes=g.nodes, initializers=g.initializers, inputs=g.inputs + [ox.ValueInfo("extra", ox.FLOAT, (1,))],
                              outputs=g.outputs))
    with pytest.raises(UnsupportedModelError, match="2 inputs"):
        recognise(three)


def _edit(style, fn):
    import copy
    m = copy.deepcopy(synth.build_gcn_model(synth.GCNConfig(**spec.SMALL), seed=4, style=style))
    fn(m.graph)
    return m


@pytest.mark.parametrize("style", ["compact", "tf2onnx"])
def test_normalisation_subgraph_is_verified_not_assumed(style):
    """ADVICE r1: a model whose adjacency normalisation is not D (A - diag A + I) D must be rejected, not silently mis-computed.
    The loader evaluates the sub-graph on probe maps, so the lowering does not matter but the function does."""
    def keep_diagonal(g):                      # A_hat = A + I   (no diagonal removal)
        for n in g.nodes:
            if n.op_type == "Add" and n.outputs[0].endswith("A_hat"):
                n.inputs[0] = "cmap"

    def column_sum(g):                         # degrees from column sums: differs for non-symmetric maps
        g.initializers["const_axes_1b"] = np.array([1], np.int64)
        for n in g.nodes:
            if n.op_type == "ReduceSum" and n.outputs[0].endswith("rowsum"):
                n.inputs[1] = "const_axes_1b"

    def no_sqrt_eps(g):                        # d = 1 / (eps + rowsum)
        for n in g.nodes:
            if n.op_type == "Sqrt":
                n.op_type = "Identity"
    with pytest.raises(UnsupportedModelError, match="D \\(A - diag"):
        recognise(_edit(style, keep_diagonal))
    with pytest.raises(UnsupportedModelError, match="D \\(A - diag"):
        recognise(_edit(style, column_sum))
    with pytest.raises(UnsupportedModelError):
        recognise(_edit(style, no_sqrt_eps))
    assert recognise(_edit(style, lambda g: None)).kind == "gcn"


def test_lstm_optional_inputs():
    """tf2onnx emits initial_h / initial_c (zeros) and may emit sequence_lens: accepted when they are what the fused kernel
    assumes (zero state, full length - checked by evaluating them on probe sequences), rejected otherwise."""
    def nonzero_state(g):
        g.initializers["lm/zero_state"] = np.full_like(g.initializers["lm/zero_state"], 0.25)
    with pytest.raises(UnsupportedModelError, match="non-zero initial state"):
        recognise(_edit("tf2onnx", nonzero_state))

    def full_length_seq_lens(g):               # sequence_lens = Shape(seq)[1:2] cast to int32
        g.initializers["c1"] = np.array([1], np.int64)
        g.initializers["c2"] = np.array([2], np.int64)
        first = next(i for i, n in enumerate(g.nodes) if n.op_type == "LSTM")
        g.nodes.insert(first, ox.Node("Shape", ["seq"], ["lm/seq_shape"], name="Shape__sl"))
        g.nodes.insert(first + 1, ox.Node("Slice", ["lm/seq_shape", "c1", "c2"], ["lm/L64"], name="Slice__sl"))
        g.nodes.insert(first + 2, ox.Node("Cast", ["lm/L64"], ["lm/seq_lens"], name="Cast__sl", attrs={"to": ox.INT32}))
        for n in g.nodes:
            if n.op_type == "LSTM":
                n.inputs[4] = "lm/seq_lens"
    assert recognise(_edit("tf2onnx", full_length_seq_lens)).lstm_hidden == spec.SMALL["lstm_hidden"]

    def short_seq_lens(g):
        g.initializers["lm/three"] = np.array([3], np.int32)
        for n in g.nodes:
            if n.op_type == "LSTM":
                n.inputs[4] = "lm/three"
    with pytest.raises(UnsupportedModelError, match="sequence_lens"):
        recognise(_edit("tf2onnx", short_seq_lens))


def test_gemm_head_is_recognised():
    """tf2onnx fuses MatMul + Add on 2-D inputs into Gemm (here with transB): same plan."""
    cfg = synth.GCNConfig(**spec.SMALL)
    w = synth.make_weights(cfg, seed=4)
    base = recognise(synth.build_gcn_model(cfg, w))

    def gemm(g):
        for lname, wname, bname in (("dense", "dense_W", "dense_b"), ("labels/dense", "labels_W", "labels_b")):
            mm = next(n for n in g.nodes if n.op_type == "MatMul" and n.inputs[1] == wname)
            add = next(n for n in g.nodes if n.op_type == "Add" and mm.outputs[0] in n.inputs)
            g.initializers[wname + "_T"] = np.ascontiguousarray(g.initializers[wname].T)
            g.nodes[g.nodes.index(mm)] = ox.Node("Gemm", [mm.inputs[0], wname + "_T", bname], [add.outputs[0]], name="Gemm_" + lname,
                                                 attrs={"transB": 1})
            g.nodes.remove(add)
    import copy
    m = copy.deepcopy(synth.build_gcn_model(cfg, w))
    gemm(m.graph)
    plan = recognise(m)
    assert plan.fc_dim == base.fc_dim and plan.n_terms == base.n_terms
    for role in ("fc_W", "fc_b", "out_W", "out_b"):
        assert np.array_equal(plan.tensor(role), base.tensor(role)), role


def heads_share_lm():
    a = synth.make_weights(synth.GCNConfig(n_terms=489), seed=1)
    b = synth.make_weights(synth.GCNConfig(n_terms=320), seed=2)
    return a, b


def test_heads_share_language_model():
    a, b = heads_share_lm()
    pa = recognise(synth.build_gcn_model(synth.GCNConfig(n_terms=489), a))
    pb = recognise(synth.build_gcn_model(synth.GCNConfig(n_terms=320), b))
    assert pa.lm_fingerprint == pb.lm_fingerprint and not np.array_equal(pa.tensor("fc_W")[:100], pb.tensor("fc_W")[:100])
    c = dict(a)
    c["lstm2_R"] = a["lstm2_R"] + np.float32(1e-3)
    assert recognise(synth.build_gcn_model(synth.GCNConfig(n_terms=489), c)).lm_fingerprint != pa.lm_fingerprint


@pytest.mark.parametrize("tag", ["small", "small_relu_bias"])
def test_oracle_matches_layer_equations_and_golden(tag, model_dir, gcn_golden):
    kw, seed, n, lo, hi = spec.GCN_CASES[tag]
    cfg = synth.GCNConfig(**kw)
    w = synth.make_weights(cfg, seed)
    p = go.Predictor(model_dir[tag])
    wl = golden_workload(tag)
    for i in range(n):
        cm = co.build_align_contact_map(wl.gapped_query[i], wl.gapped_target[i], wl.coords[i], spec.THRESHOLD, spec.GEN)
        y = p.forward_pass(wl.query_seqs[i], cm)
        assert y.dtype == np.float32 and y.shape == (cfg.n_terms,)
        assert np.abs(y - deepfri_numpy(w, cfg, wl.query_seqs[i], cm)).max() < 2e-5
        assert np.abs(y - gcn_golden[tag + "_scores"][i]).max() < 1e-6


def test_oracle_full_size_golden(model_dir, gcn_golden):
    p = go.Predictor(model_dir["mf"])
    wl = golden_workload("mf")
    cm = co.build_align_contact_map(wl.gapped_query[0], wl.gapped_target[0], wl.coords[0], spec.THRESHOLD, spec.GEN)
    assert np.abs(p.forward_pass(wl.query_seqs[0], cm) - gcn_golden["mf_scores"][0]).max() < 1e-6
