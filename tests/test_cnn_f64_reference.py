"""CPU tests of the float64 DeepCNN reference (`oracle/cnn_f64.py`) that tests/test_gpu_cnn_shapes.py holds the tensor-core
kernel to, and of the shape matrix it runs on (spec.CNN_SHAPES).

- The batched reference (R64) equals the loop form `deepcnn_f64` and the fp32 ONNX interpreter on small shapes, with Keras,
  SAME_LOWER and skewed pads, without BatchNormalization, conv bias or head bias, and with a negative BN scale.
- Its fp16 mode (R16) rounds the conv weights and nothing else.
- Every defect of `cnn_f64.MUTANTS` moves the pooled features by at least 10 x the GPU test's pooled-vs-R16 bound, on the
  shape that claims the branch: the bound would catch it.
- Every shape reaches the branch it claims: the create-time arithmetic of `mdf_cnn_model_create` (csrc/cnn_tc.cu), restated
  here, gives the claimed k-blocks, zero steps, window and filter blocks, and the loader reads the plan the reference
  assumes.  The refused shapes exceed exactly one of the kernel's limits."""
import os

import numpy as np
import pytest

import cnn_f64
import gcn_oracle as go
import spec
from conftest import recognise
from metagenomic_deepfri_b200 import onnx_lite as ox
from metagenomic_deepfri_b200 import synth

MAX_CONV, MAX_ITEMS, WIN = 32, 256, 256          # MDF_MAX_CONV, CNN_MAX_ITEMS, CNN_WIN (csrc/cnn_tc.cu)


# ----------------------------------------------------------------------------------------------------------- restated arithmetic
def kernel_plan(widths, filters, pads, n_terms):
    """What mdf_cnn_model_create computes from a model's shape (csrc/cnn_tc.cu).  K = 16 steps of a conv: (plane 0, k) +
    (plane 1, k) per position, (plane 2, k) + (plane 2, k + 1) per two positions, (plane 3, 4q) + (plane 3, 4q + 4) per
    eight; a missing partner is a zero column; a k-block is four steps, padded with all-zero steps."""
    convs = []
    for w, F, pl in zip(widths, filters, pads):
        q = (w + 3) // 4
        steps = w + (w + 1) // 2 + (q + 1) // 2
        kb = (steps + 3) // 4
        convs.append(dict(w=w, F=F, pl=pl, steps=steps, kb=kb, zero_steps=4 * kb - steps, plane2_zero=w % 2 == 1,
                          plane3_zero=q % 2 == 1, pr=q * 4 - 1 - pl, plane3_reach=q * 4))
    pl_max = max(c["pl"] for c in convs)
    pr_max = max(c["pr"] for c in convs)
    gate = all(1 <= c["w"] <= 128 and c["F"] >= 128 and c["F"] % 128 == 0 and 0 <= c["pl"] < c["w"] for c in convs)
    n_items = sum(c["F"] for c in convs) // 128
    window = 128 + pl_max + pr_max + 1
    return dict(convs=convs, pl_max=pl_max, pr_max=pr_max, window=window, n_items=n_items, Ctot=sum(filters),
                item_fb_max=max(c["F"] // 128 for c in convs) - 1, ld=(2 * n_terms + 3) // 4 * 4, head_rows=2 * n_terms,
                accepted=gate and len(convs) <= MAX_CONV and n_items <= MAX_ITEMS and window <= WIN)


def _plan_of(cfg):
    return kernel_plan(cfg.filter_lens, cfg.num_filters, cnn_f64.pad_left(cfg), cfg.n_terms)


def test_kernel_plan_arithmetic():
    """The restatement on hand-counted widths: w = 1 is 3 steps (one k-block, one all-zero step); w = 2 and 9 fill their
    k-blocks exactly; w = 128 is 128 + 64 + 16 = 208 steps = 52 k-blocks."""
    p = kernel_plan((1, 2, 9, 128), (128,) * 4, (0, 0, 4, 0), 1)
    assert [c["steps"] for c in p["convs"]] == [3, 4, 16, 208]
    assert [c["kb"] for c in p["convs"]] == [1, 1, 4, 52]
    assert [c["zero_steps"] for c in p["convs"]] == [1, 0, 0, 0]
    assert p["pr_max"] == 127 and p["window"] == 128 + 4 + 127 + 1


@pytest.mark.parametrize("tag", list(spec.CNN_SHAPES))
def test_shape_matrix_reaches_its_branch(tag):
    kw, seed, edits, _ = spec.CNN_SHAPES[tag]
    cfg, w, model = spec.cnn_case(kw, seed, edits)
    p = _plan_of(cfg)
    assert p["accepted"], p
    # the loader reads the plan the reference computes: conv order, widths, pads, folded scale
    plan = recognise(model)
    assert plan.kind == "cnn" and plan.n_terms == cfg.n_terms
    assert plan.conv_width == list(cfg.filter_lens) and plan.conv_filters == list(cfg.num_filters)
    assert plan.conv_pad_left == list(cnn_f64.pad_left(cfg))
    scale, shift = cnn_f64.scale_shift(w, cfg)
    assert np.allclose(plan.tensor("scale"), scale, rtol=1e-6, atol=0)
    assert np.allclose(plan.tensor("shift"), shift, rtol=1e-5, atol=1e-6)
    kb = [c["kb"] for c in p["convs"]]
    if tag == "w1":
        c = p["convs"][0]
        assert kb == [1] and c["zero_steps"] == 1 and c["plane2_zero"] and c["plane3_zero"] and p["head_rows"] == 2
    elif tag == "narrow":
        assert sorted(set(kb)) == [1, 2, 3, 4] and p["ld"] == 8 and p["head_rows"] == 6
        fit = {c["w"] for c in p["convs"] if c["zero_steps"] == 0}
        assert {2, 9} <= fit and len(fit) < len(p["convs"])
    elif tag == "lower":
        assert "same_lower" in edits and p["window"] == WIN
        assert all(c["pl"] == c["w"] - 1 - (c["w"] - 1) // 2 for c in p["convs"])
    elif tag == "skew":
        il = max(range(3), key=lambda i: p["convs"][i]["pl"])
        ir = max(range(3), key=lambda i: p["convs"][i]["pr"])
        assert il != ir and p["window"] == 255
        assert any(c["pl"] + 1 < c["w"] - c["pl"] for c in p["convs"]) and any(c["pl"] > c["w"] - 1 - c["pl"] for c in p["convs"])
    elif tag == "edge_right":
        assert p["window"] == WIN and p["pl_max"] == 0
        assert any(c["plane3_reach"] > c["w"] for c in p["convs"])
    elif tag == "edge_left":
        assert p["window"] == WIN and p["pr_max"] == 0
        # any partner with a right reach would push the window past the limit
        assert kernel_plan(cfg.filter_lens + (2,), cfg.num_filters + (128,), cnn_f64.pad_left(cfg) + (0,), 1)["window"] > WIN
    elif tag == "conv32":
        assert len(p["convs"]) == MAX_CONV and len(set(kb)) > 8
        kinds = {(c["pl"] == (c["w"] - 1) // 2, c["pl"] == c["w"] // 2, c["pl"] == 0, c["pl"] == c["w"] - 1) for c in p["convs"]}
        assert len(kinds) >= 4
    elif tag == "items256":
        assert p["n_items"] == MAX_ITEMS and p["item_fb_max"] == 255 and p["Ctot"] == 32768
    elif tag == "mf_negbn":
        assert np.mean(scale < 0) == 0.25 and p["head_rows"] == 3886
    elif tag == "lowering":
        assert set(edits) == {"permute_concat", "no_bn", "no_conv_bias", "gemm_transB"}
        assert np.array_equal(plan.tensor("scale"), np.ones(p["Ctot"], np.float32))
        assert plan.tensor("out_b").size == 0
        assert list(cfg.filter_lens) == sorted(cfg.filter_lens, reverse=True)      # Concat order, not node order
    else:
        raise AssertionError(f"no claim checked for {tag}")


@pytest.mark.parametrize("tag", list(spec.CNN_REFUSED))
def test_refused_shapes_exceed_one_limit(tag):
    kw, seed, _ = spec.CNN_REFUSED[tag]
    cfg = synth.CNNConfig(**kw)
    p = _plan_of(cfg)
    assert not p["accepted"]
    if tag == "window257":
        assert p["window"] == WIN + 1 and p["n_items"] <= MAX_ITEMS
    if tag == "blocks257":
        assert p["n_items"] == MAX_ITEMS + 1 and p["window"] <= WIN
    if tag in ("pad_neg", "pad_w"):
        w, pl = cfg.filter_lens[0], cfg.pad_left[0]
        assert pl + (w - 1 - pl) == w - 1       # the loader's 'same' check passes: only the kernel gate can refuse it
    # the loader recognises every one of them: the refusal comes from the kernel's limits
    plan = recognise(synth.build_cnn_model(cfg, seed=seed))
    assert plan.conv_width == list(cfg.filter_lens) and plan.conv_pad_left == list(cnn_f64.pad_left(cfg))


# ----------------------------------------------------------------------------------------------------------- R64 pinned
SMALL = {
    "keras": (dict(filter_lens=(5, 8), num_filters=(128, 128), n_terms=7, logit_scale=0.5), 81, ()),
    "same_lower": (dict(filter_lens=(4, 7), num_filters=(128, 128), pad_left=(2, 3), n_terms=7, logit_scale=0.5), 82, ("same_lower",)),
    "skew": (dict(filter_lens=(6, 3, 1), num_filters=(128,) * 3, pad_left=(5, 0, 0), n_terms=7, logit_scale=0.5), 83, ()),
    "loader_edits": (dict(filter_lens=(5, 8, 2), num_filters=(128, 256, 128), n_terms=7, logit_scale=0.5), 84,
                     ("permute_concat", "no_bn", "no_conv_bias", "gemm_transB")),
}
SMALL_LENGTHS = (1, 2, 3, 7, 33, 150)


def _small_seqs(seed):
    rng = np.random.default_rng(seed)
    seqs = ["".join(rng.choice(list(spec.CNN_ALPHABET), L)) for L in SMALL_LENGTHS]
    return seqs + ["R" * 9, "AAARAAMAA", "M"]


@pytest.mark.parametrize("tag", list(SMALL))
def test_r64_matches_loop_form_and_onnx_interpreter(tag, tmp_path):
    kw, seed, edits = SMALL[tag]
    cfg, w, model = spec.cnn_case(kw, seed, edits)
    seqs = _small_seqs(seed)
    ref = cnn_f64.reference(w, cfg, seqs)
    for i, s in enumerate(seqs):
        assert np.abs(ref["scores"][i] - cnn_f64.deepcnn_f64(w, cfg, s)).max() < 1e-12, (tag, len(s))
    path = str(tmp_path / f"{tag}.onnx")
    ox.save(model, path)
    orc = go.OnnxOracle(path)
    for i, s in enumerate(seqs):
        S = go.seq2onehot(s)[None].astype(np.float32)
        pooled, labels = orc.run(["global_max_pooling1d/Max", "labels"], {"seq": S})
        assert np.abs(pooled[0] - ref["pooled"][i]).max() <= 1e-5 * max(1.0, np.abs(ref["pooled"][i]).max()), (tag, len(s))
        assert np.abs(labels[0, :, 0] - ref["scores"][i]).max() < 2e-6, (tag, len(s))
    assert np.array_equal(np.concatenate(ref["conv_pooled"], 1), ref["pooled"])


def test_r64_matches_loop_form_with_negative_bn_scale():
    cfg, w, _ = spec.cnn_case(dict(filter_lens=(8, 16), num_filters=(128, 128), n_terms=9, logit_scale=0.5), 85, ("neg_gamma",))
    scale, _ = cnn_f64.scale_shift(w, cfg)
    assert (scale < 0).sum() == 64
    seqs = _small_seqs(85)
    ref = cnn_f64.reference(w, cfg, seqs)
    for i, s in enumerate(seqs):
        assert np.abs(ref["scores"][i] - cnn_f64.deepcnn_f64(w, cfg, s)).max() < 1e-12, len(s)


def test_f16_mode_rounds_only_the_conv_weights():
    kw, seed, edits = SMALL["keras"]
    cfg, w, _ = spec.cnn_case(kw, seed, edits)
    seqs = _small_seqs(seed)
    r16 = cnn_f64.reference(w, cfg, seqs, weights="f16")
    w16 = dict(w)
    for l in range(1, len(cfg.filter_lens) + 1):
        w16[f"conv1d_{l}_W"] = w[f"conv1d_{l}_W"].astype(np.float16).astype(np.float32)
    assert np.array_equal(r16["pooled"], cnn_f64.reference(w16, cfg, seqs)["pooled"])
    d = np.abs(r16["pooled"] - cnn_f64.reference(w, cfg, seqs)["pooled"]).max()
    assert 1e-5 < d < 1e-2                 # fp16 weights: a few 1e-4 of O(1) features


def test_batch_equals_proteins_alone():
    """The vectorised batch gives each protein what it computes alone (no row of one protein leaks into another)."""
    kw, seed, edits = SMALL["skew"]
    cfg, w, _ = spec.cnn_case(kw, seed, edits)
    seqs = _small_seqs(seed)
    ref = cnn_f64.reference(w, cfg, seqs)
    for i, s in enumerate(seqs):
        assert np.array_equal(cnn_f64.reference(w, cfg, [s])["pooled"][0], ref["pooled"][i])


# ----------------------------------------------------------------------------------------------------------- sensitivity
_cases = {}


def _shape(tag):
    """(cfg, w, seqs, R16) of a matrix shape, once per session."""
    if tag not in _cases:
        kw, seed, edits, _ = spec.CNN_SHAPES[tag]
        cfg, w, _ = spec.cnn_case(kw, seed, edits)
        seqs = spec.cnn_shape_sequences(tag)
        _cases[tag] = (cfg, w, seqs, cnn_f64.reference(w, cfg, seqs, weights="f16"))
    return _cases[tag]


def test_every_mutant_has_a_claiming_shape():
    assert set(spec.CNN_MUTANT_SHAPES) == set(cnn_f64.MUTANTS)
    for tags in spec.CNN_MUTANT_SHAPES.values():
        assert tags and set(tags) <= set(spec.CNN_SHAPES)


@pytest.mark.parametrize("tag,mutant", [(t, m) for m, ts in spec.CNN_MUTANT_SHAPES.items() for t in ts])
def test_mutant_exceeds_pooled_bound(tag, mutant):
    """The reference with one defect differs from R16 by at least 10 x the GPU test's pooled-vs-R16 bound on the batch."""
    cfg, w, seqs, r16 = _shape(tag)
    mut = cnn_f64.reference(w, cfg, seqs, weights="f16", mutate=mutant)
    rms = np.sqrt(np.mean(r16["pooled"] ** 2))
    err = np.abs(mut["pooled"] - r16["pooled"]).max() / rms
    assert err >= 10 * spec.CNN_BOUNDS["pooled_r16"], f"{mutant} on {tag}: {err:.2e}"
