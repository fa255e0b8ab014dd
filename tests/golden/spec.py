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


# ---- shape matrix of the tensor-core engine (tests/test_gpu_tc_shapes.py; the float64 reference is pinned on it by
# tests/test_gcn_f64_reference.py).  tag -> (GCNConfig kwargs, model seed, long proteins, the branch the shape reaches).
# logit_scale puts at least half of the float64 reference scores of the case's batch in [0.05, 0.95] (asserted), so that
# the score comparison is not made on a saturated softmax.
TC_SHAPES = {
    "h128": (dict(lstm_hidden=128, lm_dim=256, gc_dims=(256, 256, 256), fc_dim=256, n_terms=64, logit_scale=0.01), 41, True,
             "fused LSTM generic issuer KB = 2; pair embedding, pair X.W + mean correction"),
    "h192": (dict(lstm_hidden=192, lm_dim=384, gc_dims=(384, 128), fc_dim=128, n_terms=24, logit_scale=0.02), 42, False,
             "cpg = 3; non-pair embedding with 3 n-tiles; gd 384 non-pair X.W, bn 128 adjacency"),
    "h256": (dict(lstm_hidden=256, lm_dim=512, gc_dims=(512, 384, 256, 128), fc_dim=96, n_terms=40, logit_scale=0.02), 43, False,
             "4 layers (last one in the second ping-pong buffer); mean correction after kin = 384; SIMT head (F % 64 != 0)"),
    "h320": (dict(lstm_hidden=320, lm_dim=1024, gc_dims=(128,), fc_dim=64, n_terms=1, logit_scale=0.01), 44, False,
             "cpg = 5; a single GraphConv layer; 2C = 2 in one padded head tile"),
    "h384": (dict(lstm_hidden=384, lm_dim=128, gc_dims=(640, 256), fc_dim=1024, n_terms=489, logit_scale=0.03), 45, False,
             "gd 640: 5 non-pair X.W m-tiles and 5 bn-128 adjacency tiles; mean correction with kin = 640"),
    "h448": (dict(lstm_hidden=448, lm_dim=768, gc_dims=(512, 512, 512), fc_dim=1024, n_terms=1943, logit_scale=0.03), 46, True,
             "fused LSTM KB = 7, the largest generic-issuer shape"),
    "h512_relu_bias": (dict(lstm_hidden=512, lm_dim=1024, gc_dims=(512, 512, 512), fc_dim=1024, n_terms=489, gc_activation="Relu",
                            gc_bias=True, logit_scale=0.03), 47, True,
                       "GraphConv bias and Relu in the pair-path epilogues; straight-line LSTM issuer"),
    "h64_relu_bias": (dict(lstm_hidden=64, lm_dim=128, gc_dims=(128, 384), fc_dim=100, n_terms=24, gc_activation="Relu", gc_bias=True,
                           logit_scale=0.02), 48, False,
                      "GraphConv bias and Relu on the non-pair path; SIMT head"),
}
# shapes the tensor-core engine refuses (H % 64, E % 128, GraphConv width % 128): SIMT engine only
TC_REFUSED = {
    "h96": (dict(lstm_hidden=96, lm_dim=128, gc_dims=(128, 128), fc_dim=64, n_terms=24, logit_scale=0.03), 51),
    "e192": (dict(lstm_hidden=64, lm_dim=192, gc_dims=(128, 128), fc_dim=64, n_terms=24, logit_scale=0.03), 52),
    "gc192": (dict(lstm_hidden=64, lm_dim=128, gc_dims=(192,), fc_dim=64, n_terms=24, logit_scale=0.02), 53),
}
TC_EXACT_LENGTHS = (1, 2, 3, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512, 513)
TC_LONG = (901, 1103)     # the second crosses MDF_LSTM_PRECISE_LEN (1000): the LSTM's exact weight split


def structure_batch(lengths, seed):
    """Seeded proteins of exactly these lengths with their own structures (ungapped self-alignments, 10 A, 2 generated
    contacts) -> (Workload, dense contact maps of the oracle)."""
    import numpy as np
    import cmap_oracle as co
    from metagenomic_deepfri_b200 import synth
    rng = np.random.default_rng(seed)
    lengths = [int(L) for L in lengths]
    seqs = synth.random_sequences(rng, lengths)
    coords = synth.random_walk_coords(rng, lengths)
    wl = synth.Workload(seqs, list(seqs), list(seqs), coords, THRESHOLD, GEN, f"exact_lengths_seed{seed}")
    return wl, [co.build_align_contact_map(s, s, c, THRESHOLD, GEN) for s, c in zip(seqs, coords)]


def tc_shape_lengths(seed, long=False):
    """The lengths of a shape case's main batch: the tile edges of TC_EXACT_LENGTHS, 15 random lengths in 1-400 and, for
    `long`, TC_LONG[0], in shuffled order."""
    import numpy as np
    rng = np.random.default_rng(seed)
    lengths = list(TC_EXACT_LENGTHS) + [int(L) for L in rng.integers(1, 401, 15)] + ([TC_LONG[0]] if long else [])
    rng.shuffle(lengths)
    return lengths
