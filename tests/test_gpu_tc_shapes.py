"""Both GCN engines, stage by stage, against the float64 reference (`oracle/gcn_f64.py`) at every branch of the tensor-core
engine's shape gate (spec.TC_SHAPES: hidden sizes 64 ... 512 of the fused LSTM, pair and non-pair GEMMs of one and several
tiles, 1 ... 4 GraphConv layers, Elu / Relu, with and without bias, tensor-core and SIMT heads, n_terms = 1), on proteins of
1 ... 1103 residues that sit on the 64 / 128 / 256 / 512 tile edges.

Every stage the engines expose is compared: the degree normalisation, both LSTM layers, the embedding X0, the last GraphConv
layer, every layer's pooled slice and the scores.  The tensor-core engine rounds its operands to fp16, and what matters for the
scores is the COHERENT part of that error (it survives the sum-pool; zero-mean error averages out, DESIGN.md "Precision"), so
`stage_errors` measures both the largest error and the largest per-feature mean error over a protein's residues.  Four
sensitivity controls show that these bounds catch a missing second weight term or a missing LSTM dither."""
import os
import subprocess
import sys

import numpy as np
import pytest

import gcn_f64
import spec
from metagenomic_deepfri_b200 import predict, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TOL = 1e-3               # scores, tensor-core engine (BASELINE.json north star), with the guard band around the 0.1 call threshold
TOL_SIMT = 2e-5          # scores, exact-fp32 engine, L <= 513
TOL_SIMT_LONG = 5e-5     # scores, exact-fp32 engine, L ~ 900 / 1100 (as test_gpu_configs.py's configs[3])
TAP_SIMT = 1e-4          # every per-residue stage of the exact-fp32 engine, absolute
TAPS_ON_OFF = 2e-5       # scores with the debug taps on against the path users run (taps off)
DEG_REL = 1e-6           # the degree normalisation, relative, both engines

# Tensor-core stage bounds, one per (stage, metric) for every shape: twice the worst value over the shape matrix, the long
# proteins, the batch-structure cases and the MF-shape control, measured on an NVIDIA B200 (1000 W power limit), rounded up.
#   "max": max |G - R| over a protein's residues and features, over the RMS of the stage's reference over the batch;
#   "coh": max over features of |mean over the protein's residues of (G - R)|, normalised the same way;
#   ("pool<l>", "coh"): |pooled_G - pooled_R| / L of GraphConv layer l's slice of the pooled vector, normalised by that
#   layer's reference RMS (every layer, also those without a per-residue tap);
#   "bcoh": the mean over ALL residues of the batch's proteins of >= BCOH_MIN_LEN residues (N of them) instead of one protein's,
#   times sqrt(N / 1000).  Zero-mean rounding error then reads the same at every N, as one 1000-residue protein's would, while
#   an error of the same sign in every protein - a missing weight term, an undithered LSTM - grows with N.  The per-protein
#   "coh" cannot separate those: on a 1-5-residue protein the mean over residues averages nothing and sets its bound.
TC_BOUNDS = {                                            # measured worst: value (case, length of the protein or batch)
    ("lstm1", "max"): 5.0e-3,    # 2.50e-3 (7,680 proteins of 1-48 residues at H 448, L 38)
    ("lstm1", "coh"): 1.7e-3,    # 8.12e-4 (same batch, L 1)
    ("lstm1", "bcoh"): 3.3e-4,   # 1.62e-4 (H 384, 4,568 residues)
    ("lstm2", "max"): 2.1e-2,    # 1.06e-2 (H 448, L 321)
    ("lstm2", "coh"): 5.2e-3,    # 2.56e-3 (7,680-protein batch, L 38)
    ("lstm2", "bcoh"): 7.5e-4,   # 3.73e-4 (H 384, 4,568 residues)
    ("x0", "max"): 9.2e-3,       # 4.58e-3 (7,680-protein batch, L 37)
    ("x0", "coh"): 2.3e-3,       # 1.13e-3 (7,680-protein batch, L 3)
    ("x0", "bcoh"): 5.5e-4,      # 2.71e-4 (MF shape, 8 proteins of 850-1000, 7,518 residues)
    ("gc_last", "max"): 9.2e-3,  # 4.57e-3 (H 64 Relu + bias, L 344)
    ("gc_last", "coh"): 7.8e-3,  # 3.86e-3 (7,680-protein batch, L 9)
    ("gc_last", "bcoh"): 7.9e-4,  # 3.95e-4 (H 128, 5,919 residues)
    ("pool1", "coh"): 2.9e-3,    # 1.46e-3 (H 512 Relu + bias, L 1)
    ("pool2", "coh"): 4.1e-3,    # 2.03e-3 (7,680-protein batch, L 5)
    ("pool3", "coh"): 5.4e-3,    # 2.67e-3 (7,680-protein batch, L 4)
    ("pool4", "coh"): 5.3e-3,    # 2.61e-3 (H 256, L 2)
    ("pool1", "bcoh"): 5.9e-4,   # 2.92e-4 (MF shape, 7,518 residues)
    ("pool2", "bcoh"): 6.3e-4,   # 3.11e-4 (MF shape, 7,518 residues)
    ("pool3", "bcoh"): 7.6e-4,   # 3.76e-4 (H 128, 5,919 residues)
    ("pool4", "bcoh"): 6.3e-4,   # 3.12e-4 (H 256, 3,672 residues)
}
BCOH_MIN_LEN = 256       # "bcoh" sums over the proteins of at least this many residues
RECORD = []              # (case, engine, stage, metric, worst, length of the worst protein): what the bounds were calibrated from


def _residues(taps, rows):
    """Rows of the taps' per-residue arrays that hold the proteins `rows`, in that order."""
    off = taps["off"]
    if len(rows) == len(off) - 1:
        return slice(None)
    return np.concatenate([np.arange(off[p], off[p + 1]) for p in rows])


def stage_errors(taps, ref, cfg, rows=None):
    """{(stage, metric): normalised errors} of an engine's taps against the float64 reference, one per protein ("max", "coh")
    or one for the batch ("bcoh", empty when the batch has no protein of BCOH_MIN_LEN residues).  `rows` are the proteins of
    the taps that the reference holds, ascending (default: all of them)."""
    off = ref["off"]
    L = np.diff(off)
    rows = np.arange(len(L)) if rows is None else rows
    sel = _residues(taps, rows)
    long_p = L >= BCOH_MIN_LEN
    long_r = np.repeat(long_p, L)
    unit = np.sqrt(L[long_p].sum() * 1000.0)      # sum over N residues -> noise units of one 1000-residue protein
    out = {}
    for stage, R in (("lstm1", ref["h1"]), ("lstm2", ref["h2"]), ("x0", ref["x0"]), ("gc_last", ref["gc"][-1])):
        D = taps[stage][sel].astype(np.float64) - R
        rms = np.sqrt(np.mean(R * R))
        out[(stage, "max")] = np.maximum.reduceat(np.abs(D).max(1), off[:-1]) / rms
        out[(stage, "coh")] = np.abs(np.add.reduceat(D, off[:-1], axis=0) / L[:, None]).max(1) / rms
        out[(stage, "bcoh")] = np.array([np.abs(D[long_r].sum(0)).max() / unit / rms] if long_p.any() else [])
    goff = 0
    for l, gd in enumerate(cfg.gc_dims):
        rms = np.sqrt(np.mean(ref["gc"][l] ** 2))
        dp = taps["pooled"][rows, goff:goff + gd].astype(np.float64) - ref["pooled"][:, goff:goff + gd]
        out[(f"pool{l + 1}", "coh")] = np.abs(dp).max(1) / L / rms
        out[(f"pool{l + 1}", "bcoh")] = np.array([np.abs(dp[long_p].sum(0)).max() / unit / rms] if long_p.any() else [])
        goff += gd
    out[("deg", "rel")] = np.maximum.reduceat(np.abs(taps["deg"][sel] - ref["d"]) / ref["d"], off[:-1])
    out[("scores", "abs")] = np.abs(taps["scores"][rows].astype(np.float64) - ref["scores"]).max(1)
    return out


def run_engine(pred, engine, wl):
    """Scores of the path users run (taps off), then every tap and the scores of a run with the debug taps on."""
    pred.set_engine(engine)
    plain = pred.forward_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, spec.THRESHOLD, spec.GEN)
    pred._ctx.set_debug_taps(True)
    try:
        b = pred.upload(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords)
        try:
            pred.run(b, spec.THRESHOLD, spec.GEN)
            taps = {k: pred.fetch(b, k) for k in ("deg", "lstm1", "lstm2", "x0", "gc_last", "pooled")}
            taps["scores"] = pred.fetch_scores(b)
            taps["off"] = np.asarray(b.seq_off, np.int64)
        finally:
            b.close()
    finally:
        pred._ctx.set_debug_taps(False)
    err = float(np.abs(taps["scores"] - plain).max())
    assert err <= TAPS_ON_OFF, f"{engine}: scores with taps on differ from the plain path by {err:.2e}"
    return taps


def assert_scores(got, want, tol):
    err = float(np.abs(got - want).max()) if got.size else 0.0
    assert err <= tol, f"max |score - reference| = {err:.3e} > {tol}"
    clear = np.abs(want - 0.1) > tol
    assert np.array_equal((got >= 0.1)[clear], (want >= 0.1)[clear]), "GO calls differ outside the guard band"


def check(case, engine, taps, ref, cfg, rows=None, simt_score_tol=TOL_SIMT):
    """Every stage of one engine's run against the reference, at that engine's bounds."""
    errs = stage_errors(taps, ref, cfg, rows)
    L = np.diff(ref["off"])
    for (stage, metric), e in errs.items():
        if e.size:
            i = int(np.argmax(e))
            RECORD.append((case, engine, stage, metric, float(e[i]), int(L[i] if len(e) == len(L) else L[L >= BCOH_MIN_LEN].sum())))
    assert errs[("deg", "rel")].max() <= DEG_REL
    rows = np.arange(len(L)) if rows is None else rows
    if engine == "simt":
        sel = _residues(taps, rows)
        for stage, R in (("lstm1", ref["h1"]), ("lstm2", ref["h2"]), ("x0", ref["x0"]), ("gc_last", ref["gc"][-1])):
            assert np.abs(taps[stage][sel] - R).max() <= TAP_SIMT, stage
        goff = 0
        for l, gd in enumerate(cfg.gc_dims):
            dp = (taps["pooled"][rows, goff:goff + gd] - ref["pooled"][:, goff:goff + gd]) / L[:, None]
            assert np.abs(dp).max() <= TAP_SIMT, f"pool{l + 1}"
            goff += gd
        assert_scores(taps["scores"][rows], ref["scores"], simt_score_tol)
    else:
        bad = {k: float(errs[k].max()) for k in TC_BOUNDS if k in errs and errs[k].size and errs[k].max() > TC_BOUNDS[k]}
        assert not bad, f"{case}: tensor-core stage errors over their bounds: {bad}"
        assert_scores(taps["scores"][rows], ref["scores"], TOL)
    return errs


# ----------------------------------------------------------------------------------------------------------- fixtures
_models = {}
_refs = {}


@pytest.fixture(scope="module")
def models(tmp_path_factory):
    d = tmp_path_factory.mktemp("tc_shapes")

    def get(tag, kw, seed):
        if tag not in _models:
            path = str(d / f"{tag}.onnx")
            cfg = synth.GCNConfig(**kw)
            synth.write_gcn_model(path, cfg, seed=seed)
            _models[tag] = (predict.Predictor(path), cfg, synth.make_weights(cfg, seed))
        return _models[tag]
    yield get
    for pred, _, _ in _models.values():
        pred.close()
    _models.clear()


def reference(key, cfg, w, lengths, seed):
    """The seeded batch of these lengths and its float64 reference, computed once per key (both engines use them)."""
    if key not in _refs:
        wl, cms = spec.structure_batch(lengths, seed)
        _refs[key] = (wl, gcn_f64.reference(w, cfg, wl.query_seqs, cms))
    return _refs[key]


# ----------------------------------------------------------------------------------------------------------- the matrix
@pytest.mark.parametrize("tag", list(spec.TC_SHAPES))
@pytest.mark.parametrize("engine", ["simt", "tc"])
def test_shape_matrix(tag, engine, models):
    kw, seed, long, _ = spec.TC_SHAPES[tag]
    pred, cfg, w = models(tag, kw, seed)
    wl, ref = reference(tag, cfg, w, spec.tc_shape_lengths(seed, long), seed)
    s = ref["scores"]
    assert np.mean((s >= 0.05) & (s <= 0.95)) >= 0.5, "reference scores saturated: lower the case's logit_scale"
    taps = run_engine(pred, engine, wl)
    check(tag, engine, taps, ref, cfg, simt_score_tol=TOL_SIMT_LONG if long else TOL_SIMT)


@pytest.mark.parametrize("tag", [t for t, v in spec.TC_SHAPES.items() if v[2]])
@pytest.mark.parametrize("engine", ["simt", "tc"])
def test_long_protein_exact_split(tag, engine, models):
    """A protein over 1000 residues makes the fused LSTM use the exact (hi, lo) weight split for its whole sub-batch; alone in
    its batch, it checks that path without moving the main batch's proteins off the dithered one."""
    kw, seed, _, _ = spec.TC_SHAPES[tag]
    pred, cfg, w = models(tag, kw, seed)
    wl, ref = reference(tag + "_long", cfg, w, [spec.TC_LONG[1]], seed + 1000)
    check(tag + "_long", engine, run_engine(pred, engine, wl), ref, cfg, simt_score_tol=TOL_SIMT_LONG)


@pytest.mark.parametrize("tag", list(spec.TC_REFUSED))
def test_refused_shape_runs_on_simt(tag, models):
    kw, seed = spec.TC_REFUSED[tag]
    pred, cfg, w = models(tag, kw, seed)
    assert pred.engine == "simt"
    with pytest.raises(ValueError, match="unavailable"):
        pred.set_engine("tc")
    wl, ref = reference(tag, cfg, w, spec.tc_shape_lengths(seed), seed)
    check(tag, "simt", run_engine(pred, "simt", wl), ref, cfg)


# ----------------------------------------------------------------------------------------------------------- sensitivity controls
MF_CONTROL = dict(logit_scale=0.005)
CONTROLS = [({}, None), ({"MDF_SINGLE_TERM": "1"}, ("x0", "bcoh")), ({"MDF_SINGLE_TERM": "2"}, ("pool1", "bcoh")),
            ({"MDF_SINGLE_TERM": "4"}, ("pool2", "bcoh")), ({"MDF_LSTM_PHASES": "1"}, ("lstm2", "bcoh"))]


@pytest.mark.parametrize("env,bound", CONTROLS, ids=lambda x: ",".join(f"{k}={v}" for k, v in x.items()) or "defaults"
                         if isinstance(x, dict) else str(x and x[0]))
def test_sensitivity_controls(env, bound, monkeypatch, tmp_path):
    """On the MF shape, 8 proteins of 850 - 1000 residues (still on the dithered LSTM path): the defaults pass every bound, and
    each degraded mode (hi weight term only on one GEMM, a single LSTM dither phase) fails the bound of the stage it degrades."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    cfg = synth.GCNConfig(**MF_CONTROL)
    w = synth.make_weights(cfg, 1234)
    path = str(tmp_path / "mf.onnx")
    synth.write_gcn_model(path, cfg, seed=1234)
    lengths = [int(L) for L in np.random.default_rng(1234).integers(850, 1001, 8)]
    wl, ref = reference("mf_control", cfg, w, lengths, 1234)
    pred = predict.Predictor(path)
    try:
        taps = run_engine(pred, "tc", wl)
    finally:
        pred.close()
    name = ",".join(f"{k}={v}" for k, v in env.items()) or "mf"
    if bound is None:
        check(name, "tc", taps, ref, cfg)
        return
    errs = stage_errors(taps, ref, cfg)
    for (stage, metric), e in errs.items():
        RECORD.append((name, "tc", stage, metric, float(e.max()), int(np.diff(ref["off"]).sum())))
    assert errs[bound].max() > TC_BOUNDS[bound], f"{name}: {bound} = {errs[bound].max():.3e} does not exceed its bound"


# ----------------------------------------------------------------------------------------------------------- batch structure
def test_several_sub_batches_per_group(models):
    """H = 448 (generic issuer, KB = 7): three sub-batches of 256 proteins for every group of the fused LSTM kernel."""
    import torch
    kw, seed, _, _ = spec.TC_SHAPES["h448"]
    pred, cfg, w = models("h448", kw, seed)
    groups = torch.cuda.get_device_properties(0).multi_processor_count // (2 * cfg.lstm_hidden // 64)
    n = 3 * groups * 256
    wl, cms = spec.structure_batch([int(L) for L in np.random.default_rng(7).integers(1, 49, n)], 7)
    ref = gcn_f64.reference(w, cfg, wl.query_seqs, cms)
    check("h448_subbatches", "tc", run_engine(pred, "tc", wl), ref, cfg)


def test_more_groups_than_the_flag_area_holds(models):
    """H = 64 in CTA pairs: 148 SMs would hold 74 groups of the fused LSTM kernel, its flag area 64.  16,400 proteins are 65
    sub-batches of 256: the kernel puts the 65th on an existing group instead of refusing the batch."""
    kw, seed = spec.GCN_CASES["tc_small"][:2]
    pred, cfg, w = models("tc_small", kw, seed)
    rng = np.random.default_rng(16400)
    lengths = [int(L) for L in rng.integers(1, 17, 16400)]
    wl, cms = spec.structure_batch(lengths, 16400)
    pred.set_engine("simt")
    want = pred.forward_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, spec.THRESHOLD, spec.GEN)
    taps = run_engine(pred, "tc", wl)
    assert_scores(taps["scores"], want, TOL)
    sample = np.sort(rng.choice(len(lengths), 200, replace=False))
    ref = gcn_f64.reference(w, cfg, [wl.query_seqs[i] for i in sample], [cms[i] for i in sample])
    check("h64_16400", "tc", taps, ref, cfg, rows=sample)


def test_cluster_multicast_h256():
    """MDF_LSTM_CLUSTER=8 at H = 256 (cpg = 4) multicasts the h operand to 4 slices of a cluster (spc = 4).  The switch is read
    once per process: the H = 256 case of the matrix runs again in a child process."""
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-m", "gpu",
                        os.path.join(ROOT, "tests", "test_gpu_tc_shapes.py") + "::test_shape_matrix[tc-h256]"],
                       env=dict(os.environ, MDF_LSTM_CLUSTER="8"), cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "1 passed" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
