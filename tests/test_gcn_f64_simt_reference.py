"""CPU tests of the float64 GCN reference (`oracle/gcn_f64.py`) at the shapes only the exact-fp32 engine serves, and of the
shape matrix tests/test_gpu_simt_shapes.py runs that engine on (spec.SIMT_SHAPES).

- The reference agrees with the fp32 ONNX interpreter, every LSTM layer included, at LSTM depths 1, 3 and 4 and with eight
  GraphConv layers (test_gcn_f64_reference.py pins it at depth 2 and up to four layers).
- Every shape reaches the branch it claims: the create-time and launch arithmetic of csrc/gcn_simt.cu and mdf_model_create,
  restated here, gives the claimed CTAs per LSTM group, groups, shared memory, K tails, column passes and pooled offsets, and
  the tensor-core engine's gate (tc_model_init) refuses every shape.
- Every defect of `gcn_f64.MUTANTS` moves some stage by more than 10 x its spec.SIMT_BOUNDS bound on the shape that claims
  it: the GPU test's bounds would catch it."""
import numpy as np
import pytest

import cmap_oracle as co
import gcn_f64
import gcn_oracle as go
import spec
from metagenomic_deepfri_b200 import synth
from test_gpu_tc_shapes import stage_errors

SM_COUNT = 148                  # B200
BK, AGG_COLS = 16, 512          # sgemm_kernel's K step; graph_aggregate_kernel's columns per pass (128 threads x 4)
SMEM_LIMIT = 227 * 1024         # shared memory of one block on sm_100


# ----------------------------------------------------------------------------------------------------------- restated arithmetic
def engine_plan(cfg, lengths=(), sm_count=SM_COUNT):
    """What the exact-fp32 engine does with a model of this shape and a batch of these lengths (csrc/gcn_simt.cu): the LSTM
    launch (lstm_layer), the GEMMs with their K (simt_lstm_stack, simt_forward, head_forward), the aggregate's column passes
    and the pooled offsets; and whether each engine's gate accepts the shape."""
    H, E, gc = cfg.lstm_hidden, cfg.lm_dim, tuple(cfg.gc_dims)
    cpg = H // 16
    groups = sm_count // cpg if cpg else 0
    smem = (H * 16 * 4 + 32 * (H + 4)) * 4
    n = len(lengths)
    ng, slot = gcn_f64.lstm_groups(lengths, H, sm_count) if n else (0, np.zeros(0, np.int64))
    gemms = [("lstm_input", H)] * (cfg.lstm_layers - 1) + [("embedding", H)]
    gemms += [(f"xw{l + 1}", k) for l, k in enumerate((E,) + gc[:-1])] + [("dense", sum(gc)), ("labels", cfg.fc_dim)]
    simt_ok = (1 <= cfg.lstm_layers <= 4 and 16 <= H <= 512 and H % 16 == 0 and 1 <= len(gc) <= 8 and E > 0 and E % 4 == 0
               and all(g > 0 and g % 4 == 0 for g in gc) and cfg.fc_dim > 0 and cfg.n_terms > 0)
    tc_ok = cfg.lstm_layers == 2 and H % 64 == 0 and H <= 512 and E % 128 == 0 and all(g % 128 == 0 for g in gc)
    return dict(cpg=cpg, groups=groups, smem=smem, batch_groups=ng,
                chunks=int(slot.max()) // 32 + 1 if n else 0, k_tail={name: k % BK for name, k in gemms},
                passes=[-(-g // AGG_COLS) for g in gc], idle=[128 - min(128, g // 4) for g in gc],
                remainder=[g % AGG_COLS for g in gc], goff=list(np.cumsum((0,) + gc[:-1])),
                simt_ok=simt_ok and smem <= SMEM_LIMIT and groups >= 1, tc_ok=tc_ok)


def test_engine_plan_arithmetic():
    """The restatement on hand-counted shapes: H = 512 needs 512 x 16 x 4 + 32 x 516 floats (192.5 KiB) and leaves 4 groups;
    300 proteins over those 4 groups are 75 per group, 3 chunks of 32."""
    cfg = synth.GCNConfig(lstm_hidden=512, lstm_layers=1, lm_dim=512, gc_dims=(1028, 4))
    p = engine_plan(cfg, range(1, 301))
    assert p["smem"] == 197120 and p["groups"] == 4 and p["batch_groups"] == 4 and p["chunks"] == 3
    assert p["passes"] == [3, 1] and p["remainder"] == [4, 4] and p["idle"] == [0, 127] and p["goff"] == [0, 1028]
    assert p["k_tail"] == {"embedding": 0, "xw1": 0, "xw2": 4, "dense": 8, "labels": 0}      # dense K = 1032
    assert p["simt_ok"] and not p["tc_ok"]
    assert engine_plan(synth.GCNConfig(lstm_hidden=64, lm_dim=128, gc_dims=(128, 128)))["tc_ok"]


def test_shape_matrix_covers_the_gate():
    """Every limit mdf_model_create accepts is reached by some shape: H 16 and 512, depth 4, eight GraphConv layers, a
    width of 4 and E = 4 (more than 65535 x 64 rows: tests/test_gpu_simt_shapes.py's row-chunking batch)."""
    cfgs = [synth.GCNConfig(**kw) for kw, _, _ in spec.SIMT_SHAPES.values()]
    assert {16, 512} <= {c.lstm_hidden for c in cfgs}
    assert {1, 3, 4} <= {c.lstm_layers for c in cfgs}
    assert max(len(c.gc_dims) for c in cfgs) == 8
    assert min(min(c.gc_dims) for c in cfgs) == 4 and min(c.lm_dim for c in cfgs) == 4
    assert set(spec.SIMT_MUTANT_SHAPES) == set(gcn_f64.MUTANTS)
    for tags in spec.SIMT_MUTANT_SHAPES.values():
        assert tags and set(tags) <= set(spec.SIMT_SHAPES) | {"chunks"}


@pytest.mark.parametrize("tag", list(spec.SIMT_SHAPES))
def test_shape_matrix_reaches_its_branch(tag):
    kw, seed, _ = spec.SIMT_SHAPES[tag]
    cfg = synth.GCNConfig(**kw)
    lengths = spec.simt_shape_lengths(seed)
    p = engine_plan(cfg, lengths)
    assert p["simt_ok"] and not p["tc_ok"], p
    assert set(spec.SIMT_EXACT_LENGTHS) <= set(lengths) and len(lengths) == len(spec.SIMT_EXACT_LENGTHS) + 16
    assert spec.SIMT_LONG[0] <= max(lengths) <= spec.SIMT_LONG[1]
    tails = {k for k, v in p["k_tail"].items() if v}
    if tag == "h16_min":
        assert p["cpg"] == 1 and p["groups"] == SM_COUNT and cfg.lstm_layers == 1
        assert p["k_tail"] == {"embedding": 0, "xw1": 4, "dense": 4, "labels": 1} and p["idle"] == [127]
    elif tag == "h32_d4":
        assert cfg.lstm_layers == 4 and p["cpg"] == 2 and p["k_tail"]["xw1"] == 4 and p["k_tail"]["xw2"] == 12
    elif tag == "h48_gc8":
        assert len(cfg.gc_dims) == 8 and p["goff"] == [0, 8, 16, 24, 32, 40, 48, 56] and p["cpg"] == 3
        assert cfg.gc_activation == "Relu" and cfg.gc_bias and cfg.lstm_layers == 3
    elif tag == "h80_cols":
        assert p["cpg"] == 5 and p["passes"] == [2, 1] and p["remainder"][0] == 4 and p["k_tail"]["xw2"] == 4
    elif tag == "h144_wide":
        assert p["cpg"] == 9 and p["passes"] == [1, 3] and p["remainder"] == [60, 4]
    elif tag == "h496":
        assert p["cpg"] == 31 and p["groups"] == 4 and 186 * 1024 <= p["smem"] < 187 * 1024 and cfg.n_terms == 1943
    elif tag == "h512_d1":
        assert cfg.lstm_layers == 1 and p["smem"] == 197120 and p["smem"] <= SMEM_LIMIT
    elif tag == "h512_d4":
        assert cfg.lstm_layers == 4 and cfg.lstm_hidden == 512 and cfg.gc_dims == (512, 512, 512) and cfg.fc_dim == 1024
    elif tag == "e_wide":
        assert p["k_tail"]["xw1"] == 4 and cfg.lm_dim > 2048 and p["passes"] == [4]
    else:
        raise AssertionError(f"no claim checked for {tag}")
    assert tag in ("h512_d1", "h512_d4") or tails        # every other shape has a K tail somewhere


def test_batch_structure_cases_reach_their_branch():
    """The chunks case gives every group of the H = 512 LSTM three chunks of a time step; 148 x 33 + 5 proteins at H = 16
    give every group a second chunk, and 5 proteins leave most groups empty."""
    tag, lengths = spec.SIMT_CHUNKS
    cfg = synth.GCNConfig(**spec.SIMT_SHAPES[tag][0])
    p = engine_plan(cfg, lengths)
    assert p["batch_groups"] == 4 and p["chunks"] == 3 and len(set(lengths)) == len(lengths)
    _, slot = gcn_f64.lstm_groups(lengths, cfg.lstm_hidden, SM_COUNT)
    # a group's 33rd protein ends inside the batch's time steps: nact falls across the 32-protein chunk boundary
    L = np.asarray(lengths)
    assert L[slot == 32].min() < L.max()
    many = engine_plan(synth.GCNConfig(**spec.SIMT_SHAPES["h16_min"][0]), [5] * (SM_COUNT * 33 + 5))
    assert many["batch_groups"] == SM_COUNT and many["chunks"] == 2
    assert engine_plan(synth.GCNConfig(**spec.SIMT_SHAPES["h16_min"][0]), [5] * 5)["batch_groups"] == 5


@pytest.mark.parametrize("tag", list(spec.SIMT_REFUSED))
def test_refused_shapes_break_one_rule(tag):
    kw, _, _ = spec.SIMT_REFUSED[tag]
    p = engine_plan(synth.GCNConfig(**kw))
    assert not p["simt_ok"] and not p["tc_ok"]


# ----------------------------------------------------------------------------------------------------------- reference pinned
PIN = ["h16_min", "h48_gc8", "h32_d4"]       # LSTM depth 1; depth 3 with eight GraphConv layers, Relu + bias; depth 4
PIN_LENGTHS = (1, 2, 17, 40, 33)


def _rel(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape
    return float(np.abs(got - want).max() / max(1.0, np.abs(want).max()))


@pytest.mark.parametrize("tag", PIN)
def test_stages_match_onnx_oracle(tag, tmp_path):
    kw, seed, _ = spec.SIMT_SHAPES[tag]
    cfg = synth.GCNConfig(**kw)
    w = synth.make_weights(cfg, seed)
    path = str(tmp_path / f"{tag}.onnx")
    synth.write_gcn_model(path, cfg, seed=seed)
    oracle = go.OnnxOracle(path)
    wl, cms = spec.structure_batch(PIN_LENGTHS, seed)
    ref = gcn_f64.reference(w, cfg, wl.query_seqs, cms)
    assert len(ref["hs"]) == cfg.lstm_layers and ref["h1"] is ref["hs"][0] and ref["h2"] is ref["hs"][-1]
    act = cfg.gc_activation
    n_gc = len(cfg.gc_dims)
    nodes = [f"lm/LSTM{l}_out" for l in range(1, cfg.lstm_layers + 1)] + ["activation/Relu"] + \
            [f"GraphConv_{l}/{act}" for l in range(1, n_gc + 1)] + ["norm/d", "SumPooling/Sum", "labels"]
    off = ref["off"]
    for p, (seq, cm) in enumerate(zip(wl.query_seqs, cms)):
        L = len(seq)
        outs = dict(zip(nodes, oracle.run(nodes, {"cmap": cm[None].astype(np.float32), "seq": co.seq2onehot(seq)[None]})))
        rows = slice(off[p], off[p + 1])
        for l in range(cfg.lstm_layers):
            assert _rel(outs[f"lm/LSTM{l + 1}_out"].reshape(L, -1), ref["hs"][l][rows]) < 1e-5, (tag, p, f"lstm{l + 1}")
        assert _rel(outs["activation/Relu"].reshape(L, -1), ref["x0"][rows]) < 1e-5, (tag, p, "x0")
        for l in range(n_gc):
            assert _rel(outs[f"GraphConv_{l + 1}/{act}"].reshape(L, -1), ref["gc"][l][rows]) < 1e-5, (tag, p, f"gc{l + 1}")
        assert _rel(outs["norm/d"].reshape(L), ref["d"][rows]) < 1e-6, (tag, p, "d")
        assert _rel(outs["SumPooling/Sum"].reshape(-1), ref["pooled"][p]) < 1e-5, (tag, p, "pooled")
        assert np.abs(outs["labels"].reshape(-1, 2)[:, 0] - ref["scores"][p]).max() < 2e-6, (tag, p, "scores")


# ----------------------------------------------------------------------------------------------------------- sensitivity
_cases = {}


def _shape(tag):
    """(cfg, w, batch lengths, seqs, maps, reference) of a matrix shape or of the chunks case, once per session."""
    if tag not in _cases:
        if tag == "chunks":
            kw, seed, _ = spec.SIMT_SHAPES[spec.SIMT_CHUNKS[0]]
            lengths = spec.simt_chunk_lengths()
        else:
            kw, seed, _ = spec.SIMT_SHAPES[tag]
            lengths = spec.simt_shape_lengths(seed)
        cfg = synth.GCNConfig(**kw)
        w = synth.make_weights(cfg, seed)
        wl, cms = spec.structure_batch(lengths, seed)
        _cases[tag] = (cfg, w, wl.query_seqs, cms, gcn_f64.reference(w, cfg, wl.query_seqs, cms))
    return _cases[tag]


def as_taps(ref):
    """A reference dict in the layout of an engine's taps (what stage_errors reads)."""
    return dict(off=ref["off"], deg=ref["d"], lstm1=ref["h1"], lstm2=ref["h2"], x0=ref["x0"], gc_last=ref["gc"][-1],
                pooled=ref["pooled"], scores=ref["scores"])


def bound_ratios(errs, L):
    """{(stage, metric): worst error / its SIMT_BOUNDS bound} over the keys that have a bound."""
    out = {}
    for (stage, metric), e in errs.items():
        if not e.size or spec.simt_bound(stage, metric) is None:
            continue
        bounds = np.array([spec.simt_bound(stage, metric, int(l)) for l in L]) if len(e) == len(L) else spec.simt_bound(stage, metric)
        out[(stage, metric)] = float(np.max(e / bounds))
    return out


def test_reference_reads_as_its_own_taps():
    """The unmutated reference measured against itself is zero at every stage (the harness adds nothing)."""
    cfg, w, seqs, cms, ref = _shape("h48_gc8")
    r = bound_ratios(stage_errors(as_taps(ref), ref, cfg), np.diff(ref["off"]))
    assert r and max(r.values()) == 0.0


@pytest.mark.parametrize("tag,mutant", [(t, m) for m, ts in spec.SIMT_MUTANT_SHAPES.items() for t in ts])
def test_mutant_exceeds_a_stage_bound(tag, mutant):
    """The reference with one defect differs from the reference by more than 10 x the SIMT bound of some stage."""
    cfg, w, seqs, cms, ref = _shape(tag)
    mut = gcn_f64.reference(w, cfg, seqs, cms, mutate=mutant, sm_count=SM_COUNT)
    r = bound_ratios(stage_errors(as_taps(mut), ref, cfg), np.diff(ref["off"]))
    worst = max(r, key=r.get)
    assert r[worst] > 10, f"{mutant} on {tag}: worst {worst} at {r[worst]:.2f} x its bound"
