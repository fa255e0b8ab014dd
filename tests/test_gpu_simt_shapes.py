"""The exact-fp32 GCN engine (csrc/gcn_simt.cu), stage by stage, against the float64 reference (`oracle/gcn_f64.py`) at every
branch of mdf_model_create's gate that the tensor-core engine refuses (spec.SIMT_SHAPES: H = 16 ... 512 with cpg = H / 16 odd
and 1, 1 to 4 LSTM layers, 1 to 8 GraphConv layers, widths and E down to 4 with K tails, one to three 512-column passes of
the aggregate, the widest head), on proteins of 1 ... 1110 residues on the 32-row block edges.

Every stage the engine exposes is compared (the degree normalisation, the first and last LSTM layer, X0, the last GraphConv
layer, every layer's pooled slice and the scores) with tests/test_gpu_tc_shapes.py's `check` and `stage_errors`, and held to
spec.SIMT_BOUNDS.  The batch-structure cases split an LSTM time step into several 32-protein chunks, give the LSTM more and
fewer proteins than groups, and give the SGEMMs more rows than one launch takes.  The refused shapes raise naming the limit
they exceed.  The module prints the worst value of every (stage, metric) with its case and protein length."""
import numpy as np
import pytest

import gcn_f64
import spec
import test_gpu_tc_shapes as tcs
from metagenomic_deepfri_b200 import predict, synth

pytestmark = pytest.mark.gpu

ALONE = 1e-5             # scores of proteins run on their own against the same proteins in the big batch
WORST = {}               # (stage, metric) -> (worst value, case, protein length)


def _key(stage, metric, L):
    if stage.startswith("pool"):
        stage = "pool"
    if stage == "scores" and L >= spec.SIMT_LONG_MIN:
        stage = "scores_long"
    return stage, metric


def check_simt(case, taps, ref, cfg, rows=None):
    """tcs.check on the exact-fp32 engine (degree normalisation, absolute stage errors, scores with the guard band), then
    every (stage, metric) of stage_errors against spec.SIMT_BOUNDS; records the worst of each."""
    errs = tcs.check(case, "simt", taps, ref, cfg, rows=rows, simt_score_tol=tcs.TOL_SIMT_LONG)
    L = np.diff(ref["off"])
    long_p = L >= spec.SIMT_LONG_MIN
    bad = []
    for (stage, metric), e in errs.items():
        if spec.simt_bound(stage, metric) is None or len(e) != len(L):
            continue                                    # no SIMT bound, or one value for the batch ("bcoh")
        for part in (~long_p, long_p) if stage == "scores" else (np.ones(len(L), bool),):
            if not part.any():
                continue
            i = np.flatnonzero(part)[int(np.argmax(e[part]))]
            k = _key(stage, metric, int(L[i]))
            if k not in WORST or e[i] > WORST[k][0]:
                WORST[k] = (float(e[i]), case, int(L[i]))
            if e[i] > spec.SIMT_BOUNDS[k]:
                bad.append(f"{stage}/{metric} = {e[i]:.3e} > {spec.SIMT_BOUNDS[k]:.1e} (L {L[i]})")
    assert not bad, f"{case}: exact-fp32 stage errors over their bounds: {bad}"
    return errs


@pytest.fixture(scope="module", autouse=True)
def report(request):
    yield
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    cap = request.config.pluginmanager.get_plugin("capturemanager")
    if tr is None or cap is None or not WORST:
        return
    with cap.global_and_fixture_disabled():        # past output capture, in every report mode
        tr.write_line("")
        tr.write_line("exact-fp32 engine, worst value per (stage, metric): value (case, protein length) / bound")
        for k in sorted(WORST):
            v, case, L = WORST[k]
            tr.write_line(f"  {k[0]:>12} {k[1]:>4}: {v:.3e} ({case}, L {L}) / {spec.SIMT_BOUNDS[k]:.1e}")


_models = {}


@pytest.fixture(scope="module")
def models(tmp_path_factory):
    d = tmp_path_factory.mktemp("simt_shapes")

    def get(tag):
        if tag not in _models:
            kw, seed, _ = spec.SIMT_SHAPES[tag]
            path = str(d / f"{tag}.onnx")
            cfg = synth.GCNConfig(**kw)
            synth.write_gcn_model(path, cfg, seed=seed)
            _models[tag] = (predict.Predictor(path), cfg, synth.make_weights(cfg, seed), seed)
        return _models[tag]
    yield get
    for pred, _, _, _ in _models.values():
        pred.close()
    _models.clear()


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ----------------------------------------------------------------------------------------------------------- the matrix
@pytest.mark.parametrize("tag", list(spec.SIMT_SHAPES))
def test_shape_matrix(tag, models):
    pred, cfg, w, seed = models(tag)
    assert pred.engine == "simt"
    with pytest.raises(ValueError, match="unavailable"):
        pred.set_engine("tc")
    wl, cms = spec.structure_batch(spec.simt_shape_lengths(seed), seed)
    ref = gcn_f64.reference(w, cfg, wl.query_seqs, cms)
    s = ref["scores"]
    assert np.mean((s >= 0.05) & (s <= 0.95)) >= 0.5, "reference scores saturated: lower the case's logit_scale"
    check_simt(tag, tcs.run_engine(pred, "simt", wl), ref, cfg)


# ----------------------------------------------------------------------------------------------------------- batch structure
def test_chunks_of_a_time_step(models):
    """H = 512: 4 LSTM groups on 148 SMs; 300 proteins of lengths 1 ... 300 are 75 per group, three 32-protein chunks per
    time step, and the running count falls across the chunk boundaries as the proteins end."""
    tag = spec.SIMT_CHUNKS[0]
    pred, cfg, w, seed = models(tag)
    lengths = spec.simt_chunk_lengths()
    ng, slot = gcn_f64.lstm_groups(lengths, cfg.lstm_hidden, _sm_count())
    assert slot.max() >= 64, (ng, slot.max())
    wl, cms = spec.structure_batch(lengths, seed + 7)
    check_simt("chunks", tcs.run_engine(pred, "simt", wl), gcn_f64.reference(w, cfg, wl.query_seqs, cms), cfg)


@pytest.mark.parametrize("extra", [33, 0])
def test_groups_of_one_cta(extra, models):
    """H = 16: one CTA per group, one group per SM.  sm_count x 33 + 5 proteins give every group a second chunk (33 or 34
    proteins); 5 proteins leave all but 5 groups out of the launch."""
    pred, cfg, w, seed = models("h16_min")
    n = _sm_count() * extra + 5
    lengths = [int(L) for L in np.random.default_rng(n).integers(20, 61, n)]      # the second chunk's proteins run 20+ steps
    wl, cms = spec.structure_batch(lengths, n)
    check_simt(f"h16_n{n}", tcs.run_engine(pred, "simt", wl), gcn_f64.reference(w, cfg, wl.query_seqs, cms), cfg)


def test_more_rows_than_one_sgemm_launch(models):
    """66,000 proteins of 60-70 residues are 4.29 M rows, more than the 65535 x 64 one SGEMM launch takes: the embedding,
    X.W and their row scale and residue index continue in a second launch at row 4,194,240.  The protein that straddles that
    row, its neighbours and 64 others are compared with the reference, and with themselves run alone."""
    pred, cfg, w, seed = models("h16_min")
    rng = np.random.default_rng(66000)
    lengths = rng.integers(60, 71, 66000)
    off = np.concatenate([[0], np.cumsum(lengths)])
    assert off[-1] > spec.SIMT_MAX_ROWS
    edges = [r for r in (spec.SIMT_MAX_ROWS, 2 * spec.SIMT_MAX_ROWS) if r < off[-1]]
    straddle = [int(np.searchsorted(off, r, side="right")) - 1 for r in edges]
    assert all(off[p] < r < off[p + 1] for p, r in zip(straddle, edges))
    near = {q for p in straddle for q in (p - 1, p, p + 1)}
    others = rng.choice(np.setdiff1d(np.arange(len(lengths)), list(near)), 64, replace=False)
    sel = np.array(sorted(near | set(int(i) for i in others)))
    wl, cms = spec.structure_batch(lengths, 66000, maps_for=sel)
    taps = tcs.run_engine(pred, "simt", wl)
    assert np.array_equal(taps["off"], off)
    seqs = [wl.query_seqs[i] for i in sel]
    ref = gcn_f64.reference(w, cfg, seqs, [cms[i] for i in sel])
    check_simt("rows_4.29M", taps, ref, cfg, rows=sel)
    alone = pred.forward_structures(seqs, [wl.gapped_query[i] for i in sel], [wl.gapped_target[i] for i in sel],
                                    [wl.coords[i] for i in sel], spec.THRESHOLD, spec.GEN)
    err = float(np.abs(alone - taps["scores"][sel]).max())
    assert err <= ALONE, f"scores alone vs in the 4.29 M-row batch: {err:.2e}"


# ----------------------------------------------------------------------------------------------------------- refused shapes
@pytest.mark.parametrize("tag", list(spec.SIMT_REFUSED))
def test_refused_shape_names_its_limit(tag, tmp_path):
    kw, seed, pattern = spec.SIMT_REFUSED[tag]
    path = str(tmp_path / f"{tag}.onnx")
    synth.write_gcn_model(path, synth.GCNConfig(**kw), seed=seed)
    with pytest.raises((ValueError, NotImplementedError), match=pattern):
        predict.Predictor(path)
    # the library is left usable: a valid model still loads and runs
    kw_ok, seed_ok, _ = spec.SIMT_SHAPES["h32_d4"]
    ok = str(tmp_path / "ok.onnx")
    cfg = synth.GCNConfig(**kw_ok)
    synth.write_gcn_model(ok, cfg, seed=seed_ok)
    pred = predict.Predictor(ok)
    try:
        wl, cms = spec.structure_batch([1, 33, 70], seed_ok)
        ref = gcn_f64.reference(synth.make_weights(cfg, seed_ok), cfg, wl.query_seqs, cms)
        got = pred.forward_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, spec.THRESHOLD, spec.GEN)
        tcs.assert_scores(got, ref["scores"], tcs.TOL_SIMT)
    finally:
        pred.close()
