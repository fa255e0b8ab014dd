"""GPU tests of align-and-predict in one device job (`Predictor.submit_pairs` / `upload_pairs`, `pipeline.predict_pairs`,
`nw_trace_frame_kernel`): (query, target, coordinates) in, and everything equals the two-step route
`alignment.nw_align` -> `insert_gaps` -> `upload` / `forward_structures` - contact maps, NW scores and alignment strings bit for
bit, GO-term scores to the engines' run-to-run reproducibility."""
import numpy as np
import pytest

import cmap_oracle as co
import gcn_oracle as go
from metagenomic_deepfri_b200 import alignment, distributed, pipeline, predict, synth

pytestmark = pytest.mark.gpu
B62 = (alignment.BLOSUM62_ALPHABET, alignment.BLOSUM62)


def odd_matrix():
    """An arbitrary asymmetric matrix over a permuted alphabet that also holds 'J' (outside the GCN alphabet)."""
    rng = np.random.default_rng(5)
    alphabet = "".join(rng.permutation(list(synth.AA20 + "J")))
    return alphabet, rng.integers(-5, 8, (len(alphabet), len(alphabet))).astype(np.int8)


def walk(rng, n):
    steps = rng.normal(size=(n, 3))
    steps *= 3.8 / np.linalg.norm(steps, axis=1, keepdims=True)
    return np.round(np.cumsum(steps, axis=0), 3).astype(np.float32)


def mutate(rng, s, p_sub=0.3, p_indel=0.03):
    out = []
    for ch in s:
        u = rng.random()
        if u < p_indel:
            continue
        out.append(rng.choice(list(synth.AA20)) if u < p_indel + p_sub else ch)
        if rng.random() < p_indel:
            out.extend(rng.choice(list(synth.AA20), rng.integers(1, 6)))
    return "".join(out)


def pair_set():
    """Keyed pairs (targets = the keyed alignments' targets) + long targets (2 and 3 panels of the widest strip class) + edge
    cases: empty target, leading / trailing gaps, structures with fewer / more rows than the target, one-residue queries."""
    wl = synth.keyed_workload(np.arange(400), 9)
    qs = list(wl.query_seqs)
    ts = [g.replace("-", "") for g in wl.gapped_target]
    cs = list(wl.coords)
    rng = np.random.default_rng(3)
    for lt in (1100, 1900, 2500):
        q = "".join(rng.choice(list(synth.AA20), lt - 60))
        t = mutate(rng, q)[:lt].ljust(lt, "G")
        qs.append(q); ts.append(t); cs.append(walk(rng, lt + (7 if lt == 1900 else 0)))
    core = "MKTAYIAKQRQISFVKSHFSRQ"
    for q, t, rows in (("ACDEFG", "", 4), (core, "WWWW" + core, 26), (core, core + "WWWW", 26), ("WWWW" + core, core, 22),
                       (core + "WWWW", core, 22), (core, core, 10), (core, core[:15], 40), ("A", core, 22), ("W", "W", 1)):
        qs.append(q); ts.append(t); cs.append(walk(rng, rows))
    return qs, ts, cs


@pytest.fixture(scope="module")
def pairs():
    qs, ts, cs = pair_set()
    lt = np.array([len(t) for t in ts])
    assert (lt <= 128).any() and ((lt > 128) & (lt <= 256)).any() and ((lt > 256) & (lt <= 512)).any() and (lt > 1024).any()
    assert (lt > 2048).any()
    return qs, ts, cs


@pytest.fixture(scope="module")
def mf(model_dir):
    p = predict.Predictor(model_dir["mf"])
    yield p
    p.close()


@pytest.fixture(scope="module")
def small(model_dir):
    p = predict.Predictor(model_dir["tc_small"])
    yield p
    p.close()


def two_step(qs, ts, matrix=B62, go_=10, ge=1):
    scores, ops = alignment.nw_align(qs, ts, go_, ge, matrix)
    gapped = [alignment.insert_gaps(q, t, o) for q, t, o in zip(qs, ts, ops)]
    return scores, ops, [g[0] for g in gapped], [g[1] for g in gapped]


def test_maps_bit_identical_to_gapped_upload(mf, pairs):
    qs, ts, cs = pairs
    _, _, gq, gt = two_step(qs, ts)
    ref = mf.upload(qs, gq, gt, cs)
    fused = mf.upload_pairs(qs, ts, cs, B62)
    try:
        for thr in (6.0, 10.0):
            for gen in (0, 1, 2, 3):
                mf.run(ref, thr, gen, upto=1)
                mf.run(fused, thr, gen, upto=1)
                assert np.array_equal(mf.fetch(fused, "packed"), mf.fetch(ref, "packed")), (thr, gen)
    finally:
        ref.close()
        fused.close()


@pytest.mark.parametrize("matrix", ["blosum62", "odd"])
@pytest.mark.parametrize("gaps", [(10, 1), (0, 0), (25, 0)])
def test_alignment_outputs_equal_nw_align(mf, pairs, matrix, gaps):
    qs, ts, cs = pairs
    mat = B62 if matrix == "blosum62" else odd_matrix()
    want_s, want_ops = alignment.nw_align(qs, ts, *gaps, mat)
    _, s, ln, nm, ops = mf.forward_pairs(qs, ts, cs, mat, *gaps, alignments=True)
    assert np.array_equal(s, want_s)
    assert ops == want_ops
    assert ln.tolist() == [len(o) for o in want_ops]
    assert nm.tolist() == [o.count("M") for o in want_ops]
    b = mf.upload_pairs(qs, ts, cs, mat, *gaps)
    try:
        s2, ln2, nm2, ops2 = b.alignment(ops=True)
        assert np.array_equal(s2, want_s) and np.array_equal(ln2, ln) and np.array_equal(nm2, nm) and ops2 == want_ops
    finally:
        b.close()


@pytest.mark.parametrize("engine", ["simt", "tc"])
def test_scores_match_forward_structures(mf, pairs, engine):
    qs, ts, cs = pairs
    mf.set_engine(engine)
    try:
        _, _, gq, gt = two_step(qs, ts)
        for thr, gen in ((6.0, 2), (10.0, 0)):
            want = mf.forward_structures(qs, gq, gt, cs, thr, gen)
            got = mf.forward_pairs(qs, ts, cs, B62, threshold=thr, generated_contacts=gen)[0]
            assert np.abs(got - want).max() < 1e-5, (thr, gen)
    finally:
        mf.set_engine("tc")


def test_scores_against_oracle(mf, pairs):
    qs, ts, cs = pairs
    pick = list(range(0, 400, 40)) + [len(qs) - 9, len(qs) - 2]
    qs, ts, cs = [qs[i] for i in pick], [ts[i] for i in pick], [cs[i] for i in pick]
    _, _, gq, gt = two_step(qs, ts)
    got = mf.forward_pairs(qs, ts, cs, B62, threshold=10.0, generated_contacts=2)[0]
    oracle = go.Predictor(mf.model_path)
    want = np.stack([oracle.forward_pass(q, co.build_align_contact_map(a, b, c, 10.0, 2)) for q, a, b, c in zip(qs, gq, gt, cs)])
    assert np.abs(got - want).max() <= 1e-3
    clear = np.abs(want - 0.1) > 1e-3
    assert np.array_equal((got > 0.1)[clear], (want > 0.1)[clear])


def test_jobs_in_flight_and_stream_chunks(mf, pairs):
    qs, ts, cs = pairs
    n = len(qs)
    one = [mf.forward_pairs(qs[:200], ts[:200], cs[:200], B62), mf.forward_pairs(qs[200:], ts[200:], cs[200:], B62)]
    j1 = mf.submit_pairs(qs[:200], ts[:200], cs[:200], B62)
    j2 = mf.submit_pairs(qs[200:], ts[200:], cs[200:], B62)
    for a, b in zip(one, (j1.wait(), j2.wait())):
        assert np.abs(a[0] - b[0]).max() < 1e-5
        for x, y in zip(a[1:], b[1:]):
            assert np.array_equal(x, y)
    bounds = [(0, 150), (150, 300), (300, n)]
    out = np.full((n, mf.n_terms), -1.0, np.float32)
    chunks = ((k, hi - lo) for k, (lo, hi) in enumerate(bounds))

    def submit(k, rows):
        lo, hi = bounds[k]
        return mf.submit_pairs(qs[lo:hi], ts[lo:hi], cs[lo:hi], B62, out=rows)
    distributed.stream_chunks(submit, chunks, out)
    # each chunk against its own standalone run (same batch, so only the sum-pool atomics differ)
    want = np.concatenate([mf.forward_pairs(qs[lo:hi], ts[lo:hi], cs[lo:hi], B62)[0] for lo, hi in bounds])
    assert np.abs(out - want).max() < 1e-5


def test_predict_pairs_two_heads_align_once(mf, small, pairs):
    qs, ts, cs = pairs
    qid = [f"q{i}" for i in range(len(qs))]
    tid = [f"t{i}" for i in range(len(qs))]
    ctx = mf._ctx
    ctx.profile(True)
    try:
        scores, stats = pipeline.predict_pairs({"mf": mf, "small": small}, qid, qs, tid, ts, cs, B62, threshold=10.0)
        stages = [name for name, _, _ in ctx.profile_report()]
    finally:
        ctx.profile(False)
    assert stages.count("nw_align") == 1
    for mode, pred in (("mf", mf), ("small", small)):
        alone = pred.forward_pairs(qs, ts, cs, B62, threshold=10.0)
        assert np.abs(scores[mode] - alone[0]).max() < 1e-5, mode
    s, ops = alignment.nw_align(qs, ts, 10, 1, B62)
    assert np.array_equal(stats["nw_score"], s) and stats["n_match"].tolist() == [o.count("M") for o in ops]
    assert np.allclose(stats["identity"], [alignment._stats(o, q, t)[0] for o, q, t in zip(ops, qs, ts)])
    assert stats["target_id"] == tid


def test_errors_and_empty(mf):
    rng = np.random.default_rng(1)
    cs = [walk(rng, 5), walk(rng, 5)]
    with pytest.raises(ValueError, match="target 1 holds 'J'"):
        mf.submit_pairs(["ACDEF", "ACDEF"], ["ACDEF", "ACJEF"], cs, B62)
    with pytest.raises(ValueError, match="query 0 holds 'B'"):
        mf.submit_pairs(["ACBEF", "ACDEF"], ["ACDEF", "ACDEF"], cs, odd_matrix())
    job = mf.submit_pairs(["ACDEF", "ACJEF"], ["ACDEF", "ACDEF"], cs, odd_matrix())
    with pytest.raises(ValueError) as e:
        job.wait()
    assert str(e.value) == "Invalid character in sequence: J"
    with pytest.raises(ValueError) as want:
        mf.submit_structures(["ACDEF", "ACDEF"], ["ACDEF", "ACDEF"], ["ACDEF", "ACDEF"], [cs[0], None])
    with pytest.raises(ValueError) as got:
        mf.submit_pairs(["ACDEF", "ACDEF"], ["ACDEF", "ACDEF"], [cs[0], None], B62)
    assert str(got.value) == str(want.value)
    s, nw, ln, nm, ops = mf.forward_pairs([], [], [], B62, alignments=True)
    assert s.shape == (0, mf.n_terms) and nw.shape == ln.shape == nm.shape == (0,) and ops == []
    # the context still works after the failed submits
    assert np.isfinite(mf.forward_pairs(["ACDEF"], ["ACDEF"], cs[:1], B62)[0]).all()
