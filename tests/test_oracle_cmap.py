"""CPU tests: the contact-map oracle against the reference's own known-answer tests, the compiled
reference (oracle/_ref, when built) and the committed golden vectors."""
import os

import numpy as np
import pytest

import cmap_oracle as co

REF = co.ref_module()


def impls():
    """The port always; the reference's own compiled module only where it has been built into oracle/_ref."""
    out = [("port", co.pairwise_sqeuclidean, co.align_contact_map)]
    if REF is not None:
        out.append(("reference", REF.pairwise_sqeuclidean, REF.align_contact_map))
    return out


@pytest.mark.parametrize("name,pw,al", impls())
def test_reference_known_answers(name, pw, al):
    # mDeepFRI/tests/test_contact_map_utils.py:16-25 (values listed there; the reference forgot the assert)
    np.random.seed(42)
    m = np.random.rand(3, 3).astype(np.float32)
    exp = np.array([[0, 1.01354558, 0.12442072], [1.01354558, 0, 0.99467713], [0.12442072, 0.99467713, 0]], np.float32)
    assert np.allclose(pw(m), exp)
    # :99-110 stress case
    N = 100
    tc = np.array([[i, i + 1] for i in range(N - 1)], dtype=np.int32)
    r = al("A" * N, "A" * N, tc)
    assert r.shape == (N, N) and r[0, 1] == 1
    # :29-97 - the reference's expected matrices assume a symmetric write; the current code writes one
    # direction only (contact_map_utils.pyx:105-115; SURVEY.md §0.3).  With the symmetric sparse input the
    # pipeline really produces (np.argwhere on a symmetric map) the documented expectations hold:
    sym = lambda a: np.concatenate([a, a[:, ::-1]]).astype(np.int32)
    assert np.array_equal(al("AB", "AB", sym(np.array([[0, 1]]))), np.ones((2, 2), np.int32))
    assert np.array_equal(al("A-C", "ABC", sym(np.array([[0, 1], [1, 2], [0, 2]]))), np.ones((2, 2), np.int32))
    assert np.array_equal(al("ABC", "A-C", sym(np.array([[0, 1]])), generated_contacts=1), np.ones((3, 3), np.int32))
    # and the one-directional behaviour of the code as shipped:
    assert np.array_equal(al("AB", "AB", np.array([[0, 1]], np.int32)), np.array([[1, 1], [0, 1]], np.int32))


def test_three_point_map():
    # mDeepFRI/tests/test_conctact_map.py:36-41
    coords = np.array([[0, 0, 0], [5, 0, 0], [10, 0, 0]], np.float32)
    assert np.array_equal(co.calculate_contact_map(coords, 6.0), [[1, 1, 0], [1, 1, 1], [0, 1, 1]])
    # :20-28
    assert np.allclose(np.sqrt(co.pairwise_sqeuclidean(np.array([[0, 0, 0], [1, 1, 1]], np.float32))),
                       [[0, np.sqrt(3)], [np.sqrt(3), 0]])


def test_threshold_is_strict_and_float32():
    # bio_utils.py:214-220 under NumPy-2 weak-scalar promotion (SURVEY.md §8a a2)
    d = np.array([36.0, 35.999996, 36.000004], np.float32)
    assert list(d < co.threshold_sq(6)) == [False, True, False]
    x = np.array([[0, 0, 0], [6, 0, 0], [0, 5.9999995, 0]], np.float32)
    cm = co.calculate_contact_map(x, 6)
    assert cm[0, 1] == 0 and cm[0, 2] == 1


def test_port_matches_golden(cmap_golden):
    g = cmap_golden
    for k in range(int(g["n_cases"])):
        q, t = g[f"c{k}_q"].tobytes().decode(), g[f"c{k}_t"].tobytes().decode()
        coords = g[f"c{k}_coords"]
        thr, gen = g[f"c{k}_thr_gen"]
        thr = int(thr) if thr == int(thr) and k % 3 == 2 else float(thr)
        assert np.array_equal(co.pairwise_sqeuclidean(coords), g[f"c{k}_D"])
        sp = co.calculate_contact_map(coords, thr, "sparse") if len(coords) else np.zeros((0, 2), np.int32)
        assert np.array_equal(sp, g[f"c{k}_sparse"])
        assert np.array_equal(co.align_contact_map(q, t, sp, int(gen)), g[f"c{k}_aligned"])
        assert np.array_equal(co.pairwise_sqeuclidean_np(coords), g[f"c{k}_D"])


def test_port_matches_reference_random():
    """The port on spec.cmap_random_cases() (up to 300 residues, generated contacts 0-3, arbitrary sparse input, several
    threads) against the stored tests/golden/cmap_random_golden.npz, bit for bit; with the reference built, the
    reference against the same file."""
    import hashlib
    import spec
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cmap_random_golden.npz"))
    digest = lambda a: np.frombuffer(hashlib.blake2b(np.ascontiguousarray(a).tobytes(), digest_size=16).digest(), np.uint8)
    impls = [("port", lambda c: co.pairwise_sqeuclidean(c, threads=3),
              lambda c, thr: co.calculate_contact_map(c, thr, "sparse"),
              lambda q, t, sp, gen: co.align_contact_map(q, t, sp, gen, threads=2))]
    if REF is not None:
        impls.append(("reference", lambda c: REF.pairwise_sqeuclidean(c, 2),
                      lambda c, thr: np.argwhere(REF.pairwise_sqeuclidean(c) < co.threshold_sq(thr)).astype(np.int32),
                      lambda q, t, sp, gen: REF.align_contact_map(q, t, sp, gen, 2)))
    cases = spec.cmap_random_cases()
    assert len(cases) == int(g["n_cases"])
    for k, (gq, gt, c, thr, sp_in, gen) in enumerate(cases):
        assert np.array_equal(digest(c), g[f"r{k}_coords"]), f"case {k}: the generated inputs changed"
        Lq = int(g[f"r{k}_Lq"])
        want = np.unpackbits(g[f"r{k}_aligned"], count=Lq * Lq).reshape(Lq, Lq)
        for name, pw, sparse, al in impls:
            D = pw(c)
            assert np.array_equal(D.ravel()[g[f"r{k}_D_idx"]], g[f"r{k}_D_val"]), f"{name}, case {k}: D differs"
            assert np.array_equal(digest(D), g[f"r{k}_D"]), f"{name}, case {k}: D differs"
            sp = sparse(c, thr) if sp_in is None else sp_in
            got = al(gq, gt, sp, gen)
            assert got.shape == (Lq, Lq) and np.array_equal(got, want), f"{name}, case {k}: aligned map differs"


def test_insert_gaps_dialect():
    # mDeepFRI/tests/test_alignment.py:38-45
    assert co.insert_gaps("AACT", "AAT", "MMDM") == ("AACT", "AA-T")
    assert co.insert_gaps("AAT", "AATC", "MMMI") == ("AAT-", "AATC")
    assert co.insert_gaps("AAT", "FGTC", "XXMI") == ("AAT-", "FGTC")


def test_seq2onehot_oracle_and_product():
    # mDeepFRI/tests/test_predict.py:9-33, for the oracle twin and the product's host function
    from metagenomic_deepfri_b200 import predict
    for f in (co.seq2onehot, predict.seq2onehot):
        r = f("")
        assert r.shape == (0, 26) and r.dtype == np.float32
        assert np.all(f("D") == np.array([[0, 1] + [0] * 24]))
        r = f("-DGU")
        assert r.shape == (4, 26) and np.array_equal(r.argmax(1), [0, 1, 2, 3]) and r.sum() == 4
        with pytest.raises(ValueError):
            f("J")
    with pytest.raises(UnicodeEncodeError):
        predict.seq2onehot("ACDé")


def test_synthetic_alignments_are_consistent():
    from metagenomic_deepfri_b200 import synth
    wl = synth.make_workload(50, 5, 200, seed=3)
    for q, gq, gt, c in zip(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords):
        assert len(gq) == len(gt) and gq.replace("-", "") == q
        assert len(gt.replace("-", "")) == len(c) and c.dtype == np.float32
        assert co.align_contact_map(gq, gt, np.zeros((0, 2), np.int32)).shape == (len(q), len(q))
