"""The DeepCNN tensor-core kernel (csrc/cnn_tc.cu) against the float64 reference (`oracle/cnn_f64.py`) at every branch of its
shape gate (spec.CNN_SHAPES: widths 1 ... 128, Keras / SAME_LOWER / skewed / edge pads, one-hot windows of exactly 256
residues from either side, 32 convs, 256 filter blocks, negative BN scales, n_terms 1 ... 1943, the loader's graph variants),
on proteins that sit on the 128-row tile and four-tile group edges and on plane-3 (R / M) probes.

Per shape, four metrics (bounds in spec.CNN_BOUNDS, shared with the CPU sensitivity test):
  (a) pooled vs R16 (conv weights rounded to fp16 as the kernel's host code does, the rest in float64): the conv, scale /
      shift, ReLU and max with the fp16 rounding taken out - what is left is the order of the fp32 accumulation;
  (b) pooled vs R64;
  (c) scores vs a float64 dense + softmax of the kernel's OWN pooled vector: the exact-split head alone;
  (d) scores vs R64, with the guard band around the 0.1 call.
Then the batch structure (group rounds against the SM count, groups of four proteins, proteins across groups, shuffles,
reuse of the resident block) and the refused shapes."""
import numpy as np
import pytest

import cnn_f64
import spec
from metagenomic_deepfri_b200 import onnx_lite as ox
from metagenomic_deepfri_b200 import predict, synth

pytestmark = pytest.mark.gpu
B = spec.CNN_BOUNDS
RECORD = []              # (case, metric, worst value, length of the worst protein): what the bounds were calibrated from


# ----------------------------------------------------------------------------------------------------------- fixtures
@pytest.fixture(scope="module")
def shapes(tmp_path_factory):
    d = tmp_path_factory.mktemp("cnn_shapes")
    cache = {}

    def get(tag):
        if tag not in cache:
            kw, seed, edits, _ = spec.CNN_SHAPES[tag]
            cfg, w, model = spec.cnn_case(kw, seed, edits)
            path = str(d / f"{tag}.onnx")
            ox.save(model, path)
            cache[tag] = (predict.Predictor(path), cfg, w, path)
        return cache[tag]
    yield get
    for pred, *_ in cache.values():
        pred.close()
    if RECORD:
        worst = {}
        for case, metric, v, L in RECORD:
            if metric not in worst or v > worst[metric][1]:
                worst[metric] = (case, v, L)
        print("\nCNN shape matrix, worst per metric:")
        for metric, (case, v, L) in sorted(worst.items()):
            print(f"  {metric:11s} {v:.3e}  ({case}, L {L})  bound {B[metric]:.1e}")


def run(pred, seqs):
    pred.upload_sequences(seqs)
    pred.run_sequences()
    return pred.fetch_sequences(pooled=True)


def check(case, cfg, w, seqs, scores, pooled, r16, r64):
    """The four metrics of one batch, recorded and held to their bounds."""
    L = np.array([len(s) for s in seqs])
    p = pooled.astype(np.float64)
    _, own = cnn_f64.head(p, w, cfg.n_terms)
    errs = {
        "pooled_r16": np.abs(p - r16["pooled"]).max(1) / np.sqrt(np.mean(r16["pooled"] ** 2)),
        "pooled_r64": np.abs(p - r64["pooled"]).max(1) / np.sqrt(np.mean(r64["pooled"] ** 2)),
        "head": np.abs(scores - own).max(1),
        "scores": np.abs(scores - r64["scores"]).max(1),
    }
    for metric, e in errs.items():
        i = int(np.argmax(e))
        RECORD.append((case, metric, float(e[i]), int(L[i])))
    bad = {m: f"{e.max():.3e} (L {int(L[np.argmax(e)])})" for m, e in errs.items() if e.max() > B[m]}
    assert not bad, f"{case}: over the bounds: {bad}"
    want = r64["scores"]
    clear = np.abs(want - 0.1) > B["scores"]
    assert np.array_equal((scores >= 0.1)[clear], (want >= 0.1)[clear]), f"{case}: GO calls differ outside the guard band"


def references(cfg, w, seqs):
    return cnn_f64.reference(w, cfg, seqs, weights="f16"), cnn_f64.reference(w, cfg, seqs)


# ----------------------------------------------------------------------------------------------------------- the matrix
@pytest.mark.parametrize("tag", list(spec.CNN_SHAPES))
def test_shape_matrix(tag, shapes):
    pred, cfg, w, _ = shapes(tag)
    seqs = spec.cnn_shape_sequences(tag)
    r16, r64 = references(cfg, w, seqs)
    s = r64["scores"]
    assert np.mean((s >= 0.05) & (s <= 0.95)) >= 0.5, "reference scores saturated: lower the case's logit_scale"
    scores, pooled = run(pred, seqs)
    assert scores.shape == (len(seqs), cfg.n_terms) and pooled.shape == (len(seqs), sum(cfg.num_filters))
    check(tag, cfg, w, seqs, scores, pooled, r16, r64)


# ----------------------------------------------------------------------------------------------------------- batch structure
STRUCT = "narrow"       # a cheap shape: 7 convs of widths 2 ... 9


def tiles_and_groups(lengths):
    """The kernel's work split (mdf_cnn_upload / cnn_conv_kernel): 128-residue tiles in protein order, groups of four
    consecutive tiles -> per group, the proteins of its tiles."""
    tiles = [p for p, L in enumerate(lengths) for _ in range(0, L, 128)]
    return [tiles[i:i + 4] for i in range(0, len(tiles), 4)]


def lengths_for_groups(n_groups, seed, partial=False):
    """Seeded protein lengths whose tiles fill exactly n_groups groups (the last one with 3 tiles if `partial`): four 1-tile
    proteins (group 0), a protein of 1,100 residues (tiles 4 - 12: groups 1 - 3), one of 500 (tiles 13 - 16: groups 3 and 4),
    then lengths of 1 - 600, and 1-tile proteins to close."""
    rng = np.random.default_rng(seed)
    n_tiles = 4 * n_groups - (1 if partial else 0)
    lengths = [int(L) for L in rng.integers(1, 129, 4)] + [1100, 500]
    used = 4 + 9 + 4
    while n_tiles - used > 5:
        L = int(rng.integers(1, 601))
        t = (L + 127) // 128
        if used + t > n_tiles - 1:
            continue
        lengths.append(L)
        used += t
    lengths += [int(rng.integers(1, 129)) for _ in range(n_tiles - used)]
    assert sum((L + 127) // 128 for L in lengths) == n_tiles
    return lengths


def assert_group_structure(lengths):
    groups = tiles_and_groups(lengths)
    assert any(len(set(g)) == 4 for g in groups), "no group of four different proteins"
    span = {}
    for gi, g in enumerate(groups):
        for p in g:
            span.setdefault(p, set()).add(gi)
    assert any(len(s) == 2 for s in span.values()), "no protein across two groups"
    assert any(len(s) >= 3 for s in span.values()), "no protein across three groups"
    return len(groups)


def random_seqs(rng, lengths):
    letters = np.array(list(spec.CNN_ALPHABET))
    return ["".join(rng.choice(letters, L)) for L in lengths]


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize("kind", ["rounds_partial", "sm", "sm_plus_1"])
def test_group_rounds(kind, shapes):
    """n_groups = 2 x SMs + SMs / 4 + 1 with a partial last group (three rounds, the last one partial), = SMs (one full
    round), = SMs + 1 (a second round of one group)."""
    pred, cfg, w, _ = shapes(STRUCT)
    sm = sm_count()
    n_groups = {"rounds_partial": 2 * sm + sm // 4 + 1, "sm": sm, "sm_plus_1": sm + 1}[kind]
    lengths = lengths_for_groups(n_groups, 500 + n_groups, partial=kind == "rounds_partial")
    assert assert_group_structure(lengths) == n_groups
    rng = np.random.default_rng(n_groups)
    seqs = random_seqs(rng, lengths)
    scores, pooled = run(pred, seqs)
    check(f"{STRUCT}_{kind}", cfg, w, seqs, scores, pooled, *references(cfg, w, seqs))
    if kind == "sm":
        perm = rng.permutation(len(seqs))
        s2, p2 = run(pred, [seqs[i] for i in perm])
        assert np.array_equal(p2, pooled[perm]) and np.array_equal(s2, scores[perm])


def test_single_residue_protein(shapes):
    pred, cfg, w, _ = shapes(STRUCT)
    for s in ("R", "M", "-", "A"):
        scores, pooled = run(pred, [s])
        check(f"{STRUCT}_single", cfg, w, [s], scores, pooled, *references(cfg, w, [s]))


def test_resident_block_reuse(shapes):
    """Large batch, small batch, large batch again on one Predictor: the resident block is reused, never stale."""
    pred, cfg, w, path = shapes(STRUCT)
    rng = np.random.default_rng(31)
    large = random_seqs(rng, lengths_for_groups(sm_count() + 7, 31))
    small = random_seqs(rng, [1, 129, 300, 7, 513])
    a = run(pred, large)
    b = run(pred, small)
    c = run(pred, large)
    assert np.array_equal(a[0], c[0]) and np.array_equal(a[1], c[1])
    fresh = predict.Predictor(path)
    try:
        f = run(fresh, small)
    finally:
        fresh.close()
    assert np.array_equal(b[0], f[0]) and np.array_equal(b[1], f[1])
    check(f"{STRUCT}_reuse_small", cfg, w, small, b[0], b[1], *references(cfg, w, small))


# ----------------------------------------------------------------------------------------------------------- refusals
@pytest.mark.parametrize("tag", list(spec.CNN_REFUSED))
def test_refused_shape_then_valid_model(tag, shapes, tmp_path):
    """Loading a shape the kernel cannot run raises NotImplementedError naming the limit (host-side checks at load time);
    a valid model then loads and runs on the same context."""
    kw, seed, pattern = spec.CNN_REFUSED[tag]
    path = str(tmp_path / f"{tag}.onnx")
    synth.write_cnn_model(path, synth.CNNConfig(**kw), seed=seed)
    with pytest.raises(NotImplementedError, match=pattern):
        predict.Predictor(path)
    _, cfg, w, good = shapes("w1")
    pred = predict.Predictor(good)
    try:
        seqs = ["ACDRM", "R", "M" * 200]
        scores, pooled = run(pred, seqs)
    finally:
        pred.close()
    check(f"after_{tag}", cfg, w, seqs, scores, pooled, *references(cfg, w, seqs))
