"""Shared definition of the seeded GCN golden cases (used by make_golden.py and the tests)."""
SMALL = dict(lstm_hidden=64, lm_dim=128, gc_dims=(64, 96), fc_dim=64, n_terms=24, logit_scale=0.05)

# tag -> (GCNConfig kwargs, model seed, n proteins, Lmin, Lmax)
GCN_CASES = {
    "small": (dict(**SMALL), 5, 6, 8, 90),
    "small_relu_bias": (dict(gc_activation="Relu", gc_bias=True, **SMALL), 6, 4, 8, 90),
    "mf": (dict(), 1234, 3, 40, 140),
    # smallest shape the tensor-core engine accepts (H % 64, E % 128, g % 128)
    "tc_small": (dict(lstm_hidden=64, lm_dim=128, gc_dims=(128, 128), fc_dim=64, n_terms=24, logit_scale=0.05), 8, 9, 1, 300),
}
THRESHOLD, GEN = 10.0, 2


def workload_seed(model_seed: int) -> int:
    return model_seed + 100


def cmap_random_cases():
    """Inputs of the random contact-map cases (cmap_random_golden.npz): 60 seeded structures of 1-300 residues, 6 / 10 A,
    generated contacts 0-3.  -> [(gapped_q, gapped_t, coords, threshold, sparse, gen)]; sparse is None where the case uses
    the structure's own map (np.argwhere), else arbitrary pairs: non-symmetric, out of range and negative."""
    import numpy as np
    from metagenomic_deepfri_b200 import synth
    rng = np.random.default_rng(7)
    wl = synth.make_workload(60, 1, 300, seed=9, threshold=6.0)
    out = []
    for i in range(len(wl)):
        c = wl.coords[i]
        sp = rng.integers(-3, len(c) + 5, size=(50, 2)).astype(np.int32) if i % 5 == 0 else None
        out.append((wl.gapped_query[i], wl.gapped_target[i], c, (6.0, 10.0)[i % 2], sp, i % 4))
    return out


# ---- sequence-only DeepCNN cases: tag -> (CNNConfig kwargs, model seed, n sequences, Lmin, Lmax)
CNN_CASES = {
    # odd / even widths, unequal filter counts, 1..300 residues (tiles of 128: one, two and three per protein)
    "cnn_small": (dict(filter_lens=(5, 8, 16, 33), num_filters=(128, 256, 128, 128), n_terms=24, logit_scale=0.3), 21, 12, 1, 300),
    # the trained models' shape: 16 x 512 filters of widths 8..128, MF head
    "cnn_mf": (dict(n_terms=489), 4321, 4, 30, 420),
}
# proteins of each case re-evaluated by the CPU test (the full-size model costs seconds per protein in NumPy)
CNN_GOLDEN_CHECK = {"cnn_small": range(12), "cnn_mf": (0,)}
CNN_ALPHABET = "-DGULNTKHYWCPVSOIEFXQABZRM"


def cnn_sequences(tag):
    """Seeded sequences over the full 26-letter alphabet of predict.pyx:26 (first one of length Lmin, last of length Lmax)."""
    import numpy as np
    kw, seed, n, lo, hi = CNN_CASES[tag]
    rng = np.random.default_rng(seed + 100)
    lens = rng.integers(lo, hi + 1, n)
    lens[0], lens[-1] = lo, hi
    letters = np.array(list(CNN_ALPHABET))
    return ["".join(rng.choice(letters, int(L))) for L in lens]
