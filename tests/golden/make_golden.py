"""Generates tests/golden/*.npz.  Run in the authoring container (needs /root/reference for the
contact-map half):   python tests/golden/make_golden.py

  cmap_golden.npz  - outputs of the UNMODIFIED reference (oracle/_ref: mDeepFRI/contact_map_utils.pyx
                     compiled by oracle/Makefile) + the NumPy glue of bio_utils.py:214-223.
  cmap_random_golden.npz - pairwise_sqeuclidean (several threads) and align_contact_map on spec.cmap_random_cases():
                     structures up to 300 residues, generated contacts 0-3, arbitrary sparse input.  Written from
                     the reference like cmap_golden.npz; where the reference is not built,
                     `python tests/golden/make_golden.py --cmap-random-from-port` writes this file alone from the C port
                     (oracle/cmap_oracle.c).  Its `source` entry names which one wrote it.
  gcn_golden.npz   - outputs of oracle/gcn_oracle.py (fp32 NumPy ONNX interpreter) on seeded
                     random-init models.  PARITY UNPINNED: the reference has no golden vectors for
                     Predictor and onnxruntime is not available; these pin the CUDA path and the
                     oracle against regressions only.
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import mdf_pkg  # noqa: E402

mdf_pkg.load()
from metagenomic_deepfri_b200 import synth  # noqa: E402
import cmap_oracle as co  # noqa: E402
import gcn_oracle as go  # noqa: E402

sys.path.insert(0, HERE)
import spec  # noqa: E402


def edge_cases():
    """(gapped_q, gapped_t, n_coords_delta) hand-written alignments: leading/trailing gaps,
    '-/-' columns, all-gap target, structure longer/shorter than the aligned target."""
    return [
        ("ACDEFGHIKL", "ACDEFGHIKL", 0),
        ("--ACDEFG", "LMACDEFG", 0),
        ("ACDEFG--", "ACDEFGLM", 0),
        ("ACDEFGHIK", "AC--FG-IK", 0),
        ("AC-EF-HIK", "ACDEFGHIK", 0),
        ("A-C-E", "A-CDE", 0),             # '-/-' column
        ("ACDEF", "-----", 0),             # query fully unaligned
        ("-----ACDEF", "LMNPQ-----", 0),
        ("ACDEFGHIKLMNPQ", "ACDEFGHIKLMNPQ", -5),   # structure shorter than target sequence
        ("ACDEFGHIKLMNPQ", "ACDEFGHIKLMNPQ", +4),   # structure longer
        ("A", "A", 0),
        ("A", "-", 0),
    ]


def digest(a):
    return np.frombuffer(hashlib.blake2b(np.ascontiguousarray(a).tobytes(), digest_size=16).digest(), np.uint8)


def write_cmap_random(pw, al, source):
    """What `pw(coords)` and `al(gapped_q, gapped_t, sparse, gen)` return on spec.cmap_random_cases(): D as a digest of all
    its bytes plus a seeded sample of 64 entries, the aligned maps bit-packed (np.packbits, row-major)."""
    out = {"source": np.array(source)}
    cases = spec.cmap_random_cases()
    for k, (gq, gt, coords, thr, sp, gen) in enumerate(cases):
        D = pw(coords)
        if sp is None:
            sp = np.argwhere(D < co.threshold_sq(thr)).astype(np.int32)          # bio_utils.py:220-223
        aligned = al(gq, gt, sp, gen)
        assert np.isin(aligned, (0, 1)).all()
        idx = np.random.default_rng(k).integers(0, D.size, 64)
        out[f"r{k}_coords"] = digest(coords)
        out[f"r{k}_D"] = digest(D)
        out[f"r{k}_D_idx"], out[f"r{k}_D_val"] = idx, D.ravel()[idx]
        out[f"r{k}_Lq"] = np.array(aligned.shape[0])
        out[f"r{k}_aligned"] = np.packbits(aligned.astype(bool))
    out["n_cases"] = np.array(len(cases))
    np.savez_compressed(os.path.join(HERE, "cmap_random_golden.npz"), **out)
    print("cmap_random_golden.npz:", len(cases), "cases from", source)


def main():
    if "--cmap-random-from-port" in sys.argv[1:]:
        write_cmap_random(lambda c: co.pairwise_sqeuclidean(c, threads=3),
                          lambda q, t, sp, gen: co.align_contact_map(q, t, sp, gen, threads=2),
                          "C port: oracle/cmap_oracle.c")
        return
    ref = co.ref_module()
    if ref is None:
        raise SystemExit("oracle/_ref is not built (make -C oracle ref)")
    rng = np.random.default_rng(20260101)
    out = {}
    k = 0
    cases = []
    wl = synth.make_workload(10, 5, 70, seed=42, threshold=6.0)
    for i in range(len(wl)):
        cases.append((wl.gapped_query[i], wl.gapped_target[i], wl.coords[i]))
    for gq, gt, delta in edge_cases():
        nt = sum(c != "-" for c in gt) + delta
        cases.append((gq, gt, synth.random_walk_coords(rng, [max(nt, 0) or 1])[0][:max(nt, 0)]))
    for gq, gt, coords in cases:
        coords = np.ascontiguousarray(coords, np.float32).reshape(-1, 3)
        for thr, gen in ((6.0, 2), (10.0, 1), (8, 0)):
            D = ref.pairwise_sqeuclidean(coords)
            cmap = (D < thr ** 2).astype(np.int32)            # bio_utils.py:220
            sparse = np.argwhere(cmap == 1).astype(np.int32)  # bio_utils.py:223
            aligned = ref.align_contact_map(gq, gt, sparse, gen)
            out[f"c{k}_q"] = np.frombuffer(gq.encode(), np.uint8)
            out[f"c{k}_t"] = np.frombuffer(gt.encode(), np.uint8)
            out[f"c{k}_coords"] = coords
            out[f"c{k}_thr_gen"] = np.array([thr, gen], np.float64)
            out[f"c{k}_D"] = D
            out[f"c{k}_sparse"] = sparse
            out[f"c{k}_aligned"] = aligned.astype(np.int8)
            k += 1
    out["n_cases"] = np.array(k)
    np.savez_compressed(os.path.join(HERE, "cmap_golden.npz"), **out)
    print("cmap_golden.npz:", k, "cases")
    write_cmap_random(lambda c: ref.pairwise_sqeuclidean(c, 2), lambda q, t, sp, gen: ref.align_contact_map(q, t, sp, gen, 2),
                      "reference: mDeepFRI/contact_map_utils.pyx compiled unchanged (oracle/_ref)")

    # ---- GCN golden (oracle-generated)
    g = {}
    with tempfile.TemporaryDirectory() as d:
        for tag, (kw, seed, n, lo, hi) in spec.GCN_CASES.items():
            cfg = synth.GCNConfig(**kw)
            path = os.path.join(d, tag + ".onnx")
            synth.write_gcn_model(path, cfg, seed=seed)
            p = go.Predictor(path)
            w = synth.make_workload(n, lo, hi, seed=spec.workload_seed(seed), threshold=spec.THRESHOLD)
            scores = []
            for i in range(n):
                cm = co.build_align_contact_map(w.gapped_query[i], w.gapped_target[i], w.coords[i], spec.THRESHOLD, spec.GEN)
                scores.append(p.forward_pass(w.query_seqs[i], cm))
            g[tag + "_scores"] = np.stack(scores)
    np.savez_compressed(os.path.join(HERE, "gcn_golden.npz"), **g)
    print("gcn_golden.npz:", {k: v.shape for k, v in g.items()})


if __name__ == "__main__":
    main()
