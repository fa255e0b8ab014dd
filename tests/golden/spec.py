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


def structure_batch(lengths, seed, maps_for=None):
    """Seeded proteins of exactly these lengths with their own structures (ungapped self-alignments, 10 A, 2 generated
    contacts) -> (Workload, dense contact maps of the oracle).  `maps_for`: the proteins whose maps to build (default all;
    the others get None), for batches too large to hold every dense map."""
    import numpy as np
    import cmap_oracle as co
    from metagenomic_deepfri_b200 import synth
    rng = np.random.default_rng(seed)
    lengths = [int(L) for L in lengths]
    seqs = synth.random_sequences(rng, lengths)
    coords = synth.random_walk_coords(rng, lengths)
    wl = synth.Workload(seqs, list(seqs), list(seqs), coords, THRESHOLD, GEN, f"exact_lengths_seed{seed}")
    want = range(len(seqs)) if maps_for is None else set(int(i) for i in maps_for)
    return wl, [co.build_align_contact_map(s, s, c, THRESHOLD, GEN) if i in want else None
                for i, (s, c) in enumerate(zip(seqs, coords))]


def tc_shape_lengths(seed, long=False):
    """The lengths of a shape case's main batch: the tile edges of TC_EXACT_LENGTHS, 15 random lengths in 1-400 and, for
    `long`, TC_LONG[0], in shuffled order."""
    import numpy as np
    rng = np.random.default_rng(seed)
    lengths = list(TC_EXACT_LENGTHS) + [int(L) for L in rng.integers(1, 401, 15)] + ([TC_LONG[0]] if long else [])
    rng.shuffle(lengths)
    return lengths


# ---- shape matrix of the DeepCNN tensor-core kernel (tests/test_gpu_cnn_shapes.py; the float64 reference oracle/cnn_f64.py is
# pinned and the matrix's reach is restated on the CPU by tests/test_cnn_f64_reference.py).
# tag -> (CNNConfig kwargs, model seed, graph edits (cnn_case), the branch the shape reaches).  w = width, F = filters, KB =
# 64-wide k-blocks of a conv, window = 128 + pl_max + pr_max + 1 residues of the shared-memory one-hot image (at most 256).
# logit_scale puts at least half of the float64 reference scores of the case's batch in [0.05, 0.95] (asserted).
def _cycle_pads(widths):
    """Keras, SAME_LOWER, 0, w - 1 in turn."""
    return tuple((w - 1) // 2 if i % 4 == 0 else w // 2 if i % 4 == 1 else 0 if i % 4 == 2 else w - 1 for i, w in enumerate(widths))


CNN_SHAPES = {
    "w1": (dict(filter_lens=(1,), num_filters=(128,), pad_left=(0,), n_terms=1, logit_scale=0.5), 61, (),
           "KB = 1 with an all-zero K step; plane-2 and plane-3 zero partners; 2C = 2 in one head tile"),
    "narrow": (dict(filter_lens=(2, 3, 4, 5, 7, 8, 9), num_filters=(128,) * 7, n_terms=3, logit_scale=0.4), 62, (),
               "KB 1 ... 4; exact fit (w = 2, 9) and padded k-blocks; 2C = 6 -> ld 8"),
    "lower": (dict(filter_lens=(2, 4, 6, 16, 64, 128), num_filters=(128, 256, 128, 256, 128, 256), pad_left=(1, 2, 3, 8, 32, 64),
                   n_terms=24, logit_scale=0.5), 63, ("same_lower",),
              "auto_pad SAME_LOWER (pl = w / 2); window exactly 256 (128 + 64 + 63 + 1)"),
    "skew": (dict(filter_lens=(64, 64, 1), num_filters=(128, 128, 128), pad_left=(63, 0, 0), n_terms=24, logit_scale=0.5), 64, (),
             "explicit asymmetric pads; pl_max and pr_max from different convs, window 255"),
    "edge_right": (dict(filter_lens=(128, 125), num_filters=(128, 128), pad_left=(0, 0), n_terms=24, logit_scale=0.5), 65, (),
                   "window 256 from the right; plane-3 columns reach past the kernel (w = 125)"),
    "edge_left": (dict(filter_lens=(128, 4), num_filters=(128, 128), pad_left=(127, 3), n_terms=24, logit_scale=0.5), 66, (),
                  "window 256 from the left"),
    "conv32": (dict(filter_lens=tuple(range(1, 33)), num_filters=(128,) * 32, pad_left=_cycle_pads(range(1, 33)), n_terms=40,
                    logit_scale=0.3), 67, (),
               "MDF_MAX_CONV = 32 convs: 32 K-step table offsets and channel offsets"),
    "items256": (dict(filter_lens=(3,), num_filters=(32768,), pad_left=(1,), n_terms=24, logit_scale=0.3), 68, (),
                 "256 filter blocks, item_fb up to 255 (unsigned char); head K = 32768"),
    "mf_negbn": (dict(n_terms=1943, logit_scale=0.3), 69, ("neg_gamma",),
                 "BN gamma < 0 on a quarter of the channels: negative scale in the epilogue FMA; the widest head (2C = 3886)"),
    "lowering": (dict(filter_lens=(5, 8, 16), num_filters=(128, 256, 128), n_terms=24, logit_scale=0.5), 70,
                 ("permute_concat", "no_bn", "no_conv_bias", "gemm_transB"),
                 "loader: Concat inputs out of node order, no BatchNormalization, Conv without bias, Gemm(transB = 1) head "
                 "without bias"),
}
# shapes whose load must raise NotImplementedError naming the limit: tag -> (CNNConfig kwargs, seed, message pattern)
CNN_REFUSED = {
    "w129": (dict(filter_lens=(129,), num_filters=(128,), n_terms=5), 71, r"widths 1\.\.128"),
    "f192": (dict(filter_lens=(8,), num_filters=(192,), n_terms=5), 72, r"multiple of 128"),
    "window257": (dict(filter_lens=(128, 2), num_filters=(128, 128), pad_left=(0, 1), n_terms=5), 73, r"window of 257 residues .* at most 256"),
    "blocks257": (dict(filter_lens=(1, 1), num_filters=(32768, 128), n_terms=5), 74, r"257 filter blocks .* at most 256"),
    "conv33": (dict(filter_lens=tuple(range(1, 34)), num_filters=(128,) * 33, n_terms=5), 75, r"33 parallel Conv layers: .* at most 32"),
    "pad_neg": (dict(filter_lens=(8,), num_filters=(128,), pad_left=(-1,), n_terms=5), 76, r"0 <= pad < width"),
    "pad_w": (dict(filter_lens=(8,), num_filters=(128,), pad_left=(8,), n_terms=5), 77, r"0 <= pad < width"),
}
# oracle/cnn_f64.MUTANTS -> the shapes whose batch must show it: the shape that claims the branch, and `lowering` where the
# defect can show there (it has no BatchNormalization and no conv bias: every scale is 1 and every shift 0, so the epilogue
# mutants take conv32; abs_scale changes nothing where every scale is positive: only mf_negbn has negative ones)
CNN_MUTANT_SHAPES = {
    "pad_shift": ("skew", "lowering"),
    "drop_last_position": ("narrow", "lowering"),
    "swap_24_25": ("w1", "lowering"),
    "plane3_next_residue": ("edge_right", "lowering"),
    "pad_rows": ("w1", "lowering"),
    "first_512": ("conv32", "lowering"),
    "neighbour_block_bn": ("items256", "conv32"),
    "abs_scale": ("mf_negbn",),
}
# shapes whose reference is costly (wide convs or heads): a shorter batch (cnn_shape_sequences)
CNN_WIDE = ("items256", "mf_negbn")
CNN_EXACT_LENGTHS = (1, 2, 3, 127, 128, 129, 255, 256, 257, 511, 512, 513, 640, 1000)
CNN_PROBE_POS = (0, 1, 2, 3, 126, 127, 128, 129)      # and L - 1: a single R / M on a poly-A background

# Bounds of the GPU shape matrix, shared with the CPU sensitivity test (every mutant of oracle/cnn_f64.MUTANTS must exceed
# 10 x CNN_BOUNDS["pooled_r16"]).  The bounds are to be set to twice the worst value over the matrix and the batch-structure
# cases measured on an NVIDIA B200 (the test prints the worst per metric with its shape and protein length); until then they
# are the expected orders below, NOT MEASURED on the GPU:
#   pooled_r16: max |G - R16| over a batch's pooled features / RMS of R16's pooled features
#   pooled_r64: the same against R64 (includes the fp16 rounding of the conv weights)
#   head:       max |scores - float64 dense + softmax of the kernel's own pooled vector|
#   scores:     max |scores - R64 scores| (with the +-1e-3 guard band around the 0.1 call)
CNN_BOUNDS = {
    "pooled_r16": 2e-5,    # fp32 accumulation of at most 128 exact fp16 x 1.0 products per output: ~1e-6 expected
    "pooled_r64": 2e-3,    # R64 - R16 alone (the fp16 rounding of the conv weights) is up to 8.2e-4 over the matrix (lower)
    "head": 1e-4,          # the exact hi + lo split of the dense weights: fp32-level error expected
    "scores": 1e-3,        # the north-star tolerance of every score test
}


def cnn_case(kw, seed, edits=()):
    """A DeepCNN case -> (cfg, w, model): the ONNX model with `edits` applied, and the config and weight dict the float64
    reference reads for the same function (conv order = Concat order; weights the graph does not have are left out).
      same_lower:     auto_pad SAME_LOWER instead of explicit pads (cfg.pad_left must be the SAME_LOWER pads);
      neg_gamma:      BN gamma negated on every fourth channel (1, 5, 9, ...);
      permute_concat: Concat inputs in reverse node order;
      no_bn:          no BatchNormalization node;  no_conv_bias: Convs without bias;
      gemm_transB:    Gemm(transB = 1) with the transposed weight and no bias in place of MatMul + Add."""
    import dataclasses
    import numpy as np
    from metagenomic_deepfri_b200 import synth
    cfg = synth.CNNConfig(**kw)
    w = synth.make_cnn_weights(cfg, seed)
    if "neg_gamma" in edits:
        g = w["bn_gamma"].copy()
        g[1::4] *= -1
        w["bn_gamma"] = g
    m = synth.build_cnn_model(cfg, w)
    g = m.graph
    convs = [n for n in g.nodes if n.op_type == "Conv"]
    if "same_lower" in edits:
        if cfg.pad_left != tuple(k - 1 - (k - 1) // 2 for k in cfg.filter_lens):
            raise ValueError("same_lower: cfg.pad_left is not SAME_LOWER's")
        for n in convs:
            n.attrs.pop("pads")
            n.attrs["auto_pad"] = "SAME_LOWER"
    if "no_conv_bias" in edits:
        for l, n in enumerate(convs, 1):
            del n.inputs[2:]
            del g.initializers[f"conv1d_{l}_b"]
            del w[f"conv1d_{l}_b"]
    if "no_bn" in edits:
        bn = next(n for n in g.nodes if n.op_type == "BatchNormalization")
        relu = next(n for n in g.nodes if n.op_type == "Relu")
        relu.inputs[0] = bn.inputs[0]
        g.nodes.remove(bn)
        for k in ("bn_gamma", "bn_beta", "bn_mean", "bn_var"):
            del g.initializers[k]
            del w[k]
    if "gemm_transB" in edits:
        mm = next(n for n in g.nodes if n.op_type == "MatMul")
        add = next(n for n in g.nodes if n.op_type == "Add" and mm.outputs[0] in n.inputs)
        g.initializers["labels_W_T"] = np.ascontiguousarray(w["labels_W"].T)
        g.nodes[g.nodes.index(mm)] = type(mm)("Gemm", [mm.inputs[0], "labels_W_T"], [add.outputs[0]], name="Gemm__head",
                                              attrs={"transB": 1})
        g.nodes.remove(add)
        del g.initializers["labels_W"], g.initializers["labels_b"]
        del w["labels_b"]
    if "permute_concat" in edits:
        cat = next(n for n in g.nodes if n.op_type == "Concat")
        cat.inputs.reverse()
        nc = len(convs)
        wr = {k: v for k, v in w.items() if not k.startswith("conv1d_")}
        for l in range(1, nc + 1):
            for s in ("W", "b"):
                if f"conv1d_{nc + 1 - l}_{s}" in w:
                    wr[f"conv1d_{l}_{s}"] = w[f"conv1d_{nc + 1 - l}_{s}"]
        pads = cfg.pad_left if cfg.pad_left is not None else tuple((k - 1) // 2 for k in cfg.filter_lens)
        cfg = dataclasses.replace(cfg, filter_lens=cfg.filter_lens[::-1], num_filters=cfg.num_filters[::-1], pad_left=pads[::-1])
        w = wr
    return cfg, w, m


def cnn_shape_sequences(tag):
    """The batch of a CNN_SHAPES case over the full 26-letter alphabet, in shuffled order: the tile and group edges of
    CNN_EXACT_LENGTHS, random lengths in 1-400, R / M / '-' homopolymers, a single R or M on a poly-A background at
    CNN_PROBE_POS and at L - 1, and one protein of about 2,000 residues.  The wide shapes (CNN_WIDE) get fewer and shorter
    ones, to keep their float64 reference to a few thousand residues."""
    import numpy as np
    seed = CNN_SHAPES[tag][1]
    rng = np.random.default_rng(seed + 100)
    letters = np.array(list(CNN_ALPHABET))
    wide = tag in CNN_WIDE
    lengths = [L for L in CNN_EXACT_LENGTHS if not wide or L <= 513] + [int(L) for L in rng.integers(1, 401, 5 if wide else 15)]
    if not wide:
        lengths.append(int(rng.integers(1950, 2051)))
    seqs = ["".join(rng.choice(letters, L)) for L in lengths]
    hl = 40 if wide else 150
    seqs += ["R" * hl, "M" * hl, "-" * hl]
    pl = 131
    for ch in ("RM"[:1] if wide else "RM"):
        for p in CNN_PROBE_POS + (pl - 1,):
            seqs.append("A" * p + ch + "A" * (pl - 1 - p))
    order = rng.permutation(len(seqs))
    return [seqs[i] for i in order]


# ---- shape matrix of the exact-fp32 engine (tests/test_gpu_simt_shapes.py; the float64 reference's mutants and the matrix's
# reach are restated on the CPU by tests/test_gcn_f64_simt_reference.py).  Every shape is one the tensor-core engine refuses
# and the exact-fp32 engine serves (mdf_model_create: 1-4 LSTM layers, H = 16 ... 512 in steps of 16, 1-8 GraphConv layers,
# E and every width a multiple of 4, any F and C).  tag -> (GCNConfig kwargs, model seed, the branch the shape reaches).
# cpg = H / 16 CTAs per LSTM group, 148 / cpg groups on a B200; GEMM tiles are 64 x 64 x 16 (BK = 16), the aggregate takes
# 512 columns per pass.  logit_scale puts at least half of the float64 reference scores of the case's batch in [0.05, 0.95].
SIMT_SHAPES = {
    "h16_min": (dict(lstm_hidden=16, lstm_layers=1, lm_dim=4, gc_dims=(4,), fc_dim=1, n_terms=1, logit_scale=0.03), 91,
                "cpg = 1 (148 groups of one CTA); K = 4 (X.W, dense) and 1 (labels) < BK; 127 of 128 aggregate threads idle"),
    "h32_d4": (dict(lstm_hidden=32, lstm_layers=4, lm_dim=20, gc_dims=(12, 36), fc_dim=10, n_terms=3, logit_scale=0.01), 92,
               "MDF_MAX_LSTM = 4: three input GEMMs through the shared pre buffer; K tails of 20 and 12; cpg = 2"),
    "h48_gc8": (dict(lstm_hidden=48, lstm_layers=3, lm_dim=52, gc_dims=(8,) * 8, fc_dim=24, n_terms=7, gc_activation="Relu",
                     gc_bias=True, logit_scale=0.005), 93,
                "MDF_MAX_GC = 8: eight pooled slices at offsets 0, 8 ... 56; Relu + bias; cpg = 3; 3 LSTM layers"),
    "h80_cols": (dict(lstm_hidden=80, lm_dim=100, gc_dims=(516, 4), fc_dim=40, n_terms=5, logit_scale=0.03), 94,
                 "cpg = 5; a second column pass with a 4-column remainder; K = 516 into the next layer"),
    "h144_wide": (dict(lstm_hidden=144, lm_dim=64, gc_dims=(60, 1028), fc_dim=72, n_terms=24, logit_scale=0.02), 95,
                  "cpg = 9; three column passes (1028 = 2 x 512 + 4)"),
    "h496": (dict(lstm_hidden=496, lm_dim=36, gc_dims=(100, 200, 300), fc_dim=1000, n_terms=1943, logit_scale=0.03), 96,
             "cpg = 31, 4 groups, 186 KiB of shared memory; the widest head (2C = 3886)"),
    "h512_d1": (dict(lstm_hidden=512, lstm_layers=1, lm_dim=512, gc_dims=(256,), fc_dim=128, n_terms=64, logit_scale=0.03), 97,
                "192 KiB of shared memory, the largest H; the embedding reads layer 1 directly"),
    "h512_d4": (dict(lstm_hidden=512, lstm_layers=4, n_terms=489, logit_scale=0.02), 98,
                "the deepest stack at the largest H, MF widths (E 1024, gc 512 x 3, F 1024)"),
    "e_wide": (dict(lstm_hidden=64, lm_dim=2052, gc_dims=(2048,), fc_dim=64, n_terms=24, logit_scale=0.01), 99,
               "a long-K X.W (K = 2052 = 128 x 16 + 4) with a K tail; E not a multiple of 128"),
}
# oracle/gcn_f64.MUTANTS -> the shapes whose batch must show it (tests/test_gcn_f64_simt_reference.py); "chunks" is the
# batch-structure case of SIMT_CHUNKS
SIMT_MUTANT_SHAPES = {
    "slice_edge": ("h32_d4", "h80_cols", "h496"),
    "gate_order": ("h16_min", "h512_d1"),
    "one_bias": ("h16_min", "h48_gc8"),
    "k_tail": ("h16_min", "h32_d4", "h80_cols", "e_wide"),
    "col_tail": ("h80_cols", "h144_wide"),
    "row31": ("h16_min", "h48_gc8"),
    "pool_offset": ("h48_gc8", "h496"),
    "depth_input": ("h32_d4", "h48_gc8", "h512_d4"),
    "second_chunk_stale_h": ("chunks",),
}
SIMT_EXACT_LENGTHS = (1, 2, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512, 513)
SIMT_LONG = (1090, 1110)       # one protein of about 1,100 residues per shape
# batch-structure case "chunks": H 512 (4 groups of 32 CTAs on 148 SMs), 300 proteins of lengths 1 ... 300: 75 per group,
# 3 chunks of 32 proteins per time step, and the number of running proteins crosses the chunk boundaries as they end
SIMT_CHUNKS = ("h512_d1", tuple(range(1, 301)))


def simt_chunk_lengths():
    """The chunks case's lengths in seeded shuffled order."""
    import numpy as np
    lengths = list(SIMT_CHUNKS[1])
    np.random.default_rng(SIMT_SHAPES[SIMT_CHUNKS[0]][1]).shuffle(lengths)
    return lengths
# a batch of more than 65535 x 64 rows: the SGEMMs split it into launches of at most that many rows
SIMT_MAX_ROWS = 65535 * 64

# shapes mdf_model_create (or the loader, for the depths) must refuse: tag -> (GCNConfig kwargs, seed, message pattern)
_R = dict(lm_dim=8, gc_dims=(8,), fc_dim=4, n_terms=2)
SIMT_REFUSED = {
    "h8": (dict(lstm_hidden=8, **_R), 101, r"LSTM hidden size 8 .*multiple of 16 from 16 to 512"),
    "h24": (dict(lstm_hidden=24, **_R), 102, r"LSTM hidden size 24 .*multiple of 16 from 16 to 512"),
    "h528": (dict(lstm_hidden=528, **_R), 103, r"LSTM hidden size 528 .*multiple of 16 from 16 to 512"),
    "lstm5": (dict(lstm_hidden=16, lstm_layers=5, **_R), 104, r"5 LSTM layers: .*at most 4"),
    "gc9": (dict(lstm_hidden=16, lm_dim=8, gc_dims=(4,) * 9, fc_dim=4, n_terms=2), 105, r"9 GraphConv layers: .*at most 8"),
    "gc_w6": (dict(lstm_hidden=16, lm_dim=8, gc_dims=(8, 6), fc_dim=4, n_terms=2), 106,
              r"GraphConv layer 2 has width 6: .*multiple of 4"),
    "e6": (dict(lstm_hidden=16, lm_dim=6, gc_dims=(8,), fc_dim=4, n_terms=2), 107, r"embedding width 6: .*multiple of 4"),
}

# Bounds of the exact-fp32 engine, one per (stage, metric), shared with the CPU sensitivity test (every mutant of
# oracle/gcn_f64.MUTANTS must exceed 10 x the bound of some stage on the shape that claims it).  "max" and "coh" are
# tests/test_gpu_tc_shapes.py's definitions (normalised by the RMS of the stage's reference over the batch); ("pool", "coh")
# applies to every GraphConv layer's pooled slice; scores are absolute.  The stage bounds are twice the worst value over
# SIMT_SHAPES and the batch-structure cases of tests/test_gpu_simt_shapes.py, measured on an NVIDIA B200 (1000 W power
# limit), rounded up; the scores keep the project's exact-fp32 tolerances.
SIMT_BOUNDS = {                      # measured worst: value (case, protein length)
    ("lstm1", "max"): 8.3e-6,        # 4.10e-6 (chunks, L 207)
    ("lstm1", "coh"): 1.2e-6,        # 5.96e-7 (h512_d1, L 2)
    ("lstm2", "max"): 1.2e-4,        # 5.80e-5 (h512_d4, L 161): the fourth H = 512 layer
    ("lstm2", "coh"): 8.6e-6,        # 4.27e-6 (h512_d4, L 54)
    ("x0", "max"): 3.3e-5,           # 1.61e-5 (h512_d4, L 161)
    ("x0", "coh"): 4.7e-6,           # 2.33e-6 (h512_d4, L 65)
    ("gc_last", "max"): 1.6e-5,      # 7.99e-6 (h512_d4, L 65)
    ("gc_last", "coh"): 8.7e-6,      # 4.32e-6 (e_wide, L 1)
    ("pool", "coh"): 8.7e-6,         # 4.32e-6 (e_wide, L 1)
    ("scores", "abs"): 2e-5,         # L <= 513; 5.60e-6 (h512_d4, L 513)
    ("scores_long", "abs"): 5e-5,    # L ~ 1100; 8.94e-6 (h512_d4, L 1090)
}
SIMT_LONG_MIN = 1000                 # proteins of at least this length are held to ("scores_long", "abs")


def simt_bound(stage, metric, L=0):
    """SIMT_BOUNDS entry of a stage_errors key (pool<l> -> pool; scores of a long protein -> scores_long)."""
    if stage.startswith("pool"):
        stage = "pool"
    if stage == "scores" and L >= SIMT_LONG_MIN:
        stage = "scores_long"
    return SIMT_BOUNDS.get((stage, metric))


def simt_shape_lengths(seed):
    """The lengths of a SIMT_SHAPES case's batch: the 32-row block edges of SIMT_EXACT_LENGTHS, 15 random lengths in 1-400
    and one of SIMT_LONG, in shuffled order."""
    import numpy as np
    rng = np.random.default_rng(seed)
    lengths = list(SIMT_EXACT_LENGTHS) + [int(L) for L in rng.integers(1, 401, 15)] + [int(rng.integers(SIMT_LONG[0], SIMT_LONG[1] + 1))]
    rng.shuffle(lengths)
    return lengths
