"""ORACLE — TEST INFRASTRUCTURE ONLY (never imported by the product package).

Float64 restatement of upstream DeepFRI's sequence-only DeepCNN head (parallel Conv1D over the one-hot sequence -> concat ->
conv bias + BatchNormalization -> ReLU -> max over residues -> dense -> softmax over (C, 2) pairs), written from the layer
equations, not from the ONNX graph: it takes the weight dict of `synth.make_cnn_weights(cfg, seed)` and the per-conv left
pads of `cfg.pad_left` (None: Keras 'same', (k - 1) // 2), and returns every stage.

`deepcnn_f64` is the one-protein loop form (scores only).  `reference` runs a whole batch: a conv over a one-hot input is a
product of the one-hot windows [rows, k * 26] with the weights [k * 26, F], vectorised over all residues of the batch.

  weights="f64": R64, the model as written.
  weights="f16": R16, the conv weights rounded to fp16 first (round to nearest even, as the kernel's host code does with
                 `__float2half_rn`), everything else in float64: what the tensor-core kernel computes up to the order of
                 its fp32 accumulation.
  mutate=<one of MUTANTS>: the reference with one defect of the kind the kernel's layout invites (see MUTANTS), for tests
                 that show a bound would catch it.

Missing optional weights are read as the graph without them: no `bn_*` entries = no BatchNormalization, no `conv1d_<l>_b` =
a Conv without bias, no `labels_b` = a head without bias.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence

import numpy as np

ALPHABET = "-DGULNTKHYWCPVSOIEFXQABZRM"      # predict.pyx:26; channels 24 / 25 are R / M

# defect -> what it does to the computation
MUTANTS = {
    "pad_shift": "the first conv reads its window one residue later (left pad + 1)",
    "drop_last_position": "every conv ignores its last kernel position",
    "swap_24_25": "channels 24 and 25 (R, M) trade places",
    "plane3_next_residue": "channels 24 / 25 of a kernel position are read from the next residue",
    "pad_rows": "rows L .. ceil(L / 128) * 128 - 1 of a protein's last tile enter the max",
    "first_512": "a protein of more than 512 residues is pooled over its first 512 only",
    "neighbour_block_bn": "filter block 1 (channels 128 .. 255) gets block 0's scale and shift",
    "abs_scale": "|scale| in place of scale",
}


def pad_left(cfg) -> tuple:
    """Per-conv zero residues before position 0: cfg.pad_left, or Keras 'same' ((k - 1) // 2) where it is None."""
    pl = getattr(cfg, "pad_left", None)
    return tuple(int(p) for p in pl) if pl is not None else tuple((k - 1) // 2 for k in cfg.filter_lens)


def encode(seq: str) -> np.ndarray:
    out = np.frombuffer(seq.encode("ascii"), np.uint8)
    lut = np.full(256, 255, np.uint8)
    lut[np.frombuffer(ALPHABET.encode(), np.uint8)] = np.arange(26, dtype=np.uint8)
    idx = lut[out]
    if (idx == 255).any():
        raise ValueError(f"Invalid character in sequence: {seq[int(np.argmax(idx == 255))]}")
    return idx


def scale_shift(w: Dict[str, np.ndarray], cfg):
    """Conv bias and inference-mode BatchNormalization as one per-channel affine map y = conv * scale + shift (float64)."""
    bias = np.concatenate([w[f"conv1d_{l}_b"].astype(np.float64) if f"conv1d_{l}_b" in w else np.zeros(F)
                           for l, F in enumerate(cfg.num_filters, 1)])
    if "bn_gamma" not in w:
        return np.ones_like(bias), bias
    s = w["bn_gamma"].astype(np.float64) / np.sqrt(w["bn_var"].astype(np.float64) + cfg.bn_epsilon)
    return s, (bias - w["bn_mean"].astype(np.float64)) * s + w["bn_beta"].astype(np.float64)


def head(pooled: np.ndarray, w: Dict[str, np.ndarray], n_terms: int):
    """Dense layer and softmax over (C, 2) pairs in float64 -> (logits [n, C, 2], scores [n, C])."""
    z = np.asarray(pooled, np.float64) @ w["labels_W"].astype(np.float64)
    if "labels_b" in w:
        z = z + w["labels_b"].astype(np.float64)
    z = z.reshape(len(z), n_terms, 2)
    e = np.exp(z - z.max(2, keepdims=True))
    return z, (e / e.sum(2, keepdims=True))[:, :, 0]


def deepcnn_f64(w, cfg, seq):
    """Keras semantics, loop form, one protein: Conv1D(padding='same') pads pl zeros before and k - 1 - pl after;
    BatchNormalization (inference) ; ReLU ; GlobalMaxPooling1D ; dense ; softmax over (C, 2) pairs."""
    L = len(seq)
    idx = [ALPHABET.index(ch) for ch in seq]
    feats = []
    for l, (k, pl) in enumerate(zip(cfg.filter_lens, pad_left(cfg)), 1):
        W = w[f"conv1d_{l}_W"][:, :, 0, :].astype(np.float64)       # [F, 26, k]
        b = w[f"conv1d_{l}_b"].astype(np.float64) if f"conv1d_{l}_b" in w else np.zeros(len(W))
        y = np.tile(b, (L, 1))
        for t in range(L):
            for j in range(k):
                r = t + j - pl
                if 0 <= r < L:
                    y[t] += W[:, idx[r], j]
        feats.append(y)
    x = np.concatenate(feats, axis=1)
    if "bn_gamma" in w:
        x = (x - w["bn_mean"]) / np.sqrt(w["bn_var"].astype(np.float64) + cfg.bn_epsilon) * w["bn_gamma"] + w["bn_beta"]
    p = np.maximum(x, 0).max(axis=0)
    z = (p @ w["labels_W"].astype(np.float64) + (w["labels_b"] if "labels_b" in w else 0.0)).reshape(cfg.n_terms, 2)
    e = np.exp(z - z.max(axis=1, keepdims=True))
    return (e / e.sum(axis=1, keepdims=True))[:, 0]


_COLS = 1 << 11          # filters per product: bounds the [rows, filters] float64 block of a wide conv


def reference(w: Dict[str, np.ndarray], cfg, seqs: Sequence[str], weights: str = "f64",
              mutate: Optional[str] = None) -> Dict[str, object]:
    """Every stage of the DeepCNN head for a batch, in float64:
      conv_pooled [per conv: n, F_c] (max over residues of ReLU(conv * scale + shift)), pooled [n, sum F] (concatenated
      in conv order, the layout of the kernel's pooled vector), logits [n, C, 2], scores [n, C]."""
    if weights not in ("f64", "f16"):
        raise ValueError(weights)
    if mutate is not None and mutate not in MUTANTS:
        raise ValueError(f"unknown mutant {mutate!r}")
    n = len(seqs)
    if n == 0:
        raise ValueError("empty batch")
    codes = [encode(s) for s in seqs]
    L = np.array([len(c) for c in codes], np.int64)
    if (L < 1).any():
        raise ValueError("empty sequence: the max over residues needs at least one")
    start = np.zeros(n + 1, np.int64)
    np.cumsum(L, out=start[1:])
    idx = np.concatenate(codes).astype(np.int64)
    if mutate == "swap_24_25":
        idx = np.where(idx == 24, 25, np.where(idx == 25, 24, idx))
    # output rows: t = 0 .. L - 1 of every protein (and the pad rows of its last 128-row tile for "pad_rows")
    R = (L + 127) // 128 * 128 if mutate == "pad_rows" else L
    roff = np.zeros(n + 1, np.int64)
    np.cumsum(R, out=roff[1:])
    prot = np.repeat(np.arange(n), R)
    t = np.arange(int(roff[-1])) - roff[prot]
    Lr, sr = L[prot], start[prot]
    pooled_rows = t < (np.minimum(Lr, 512) if mutate == "first_512" else (R[prot] if mutate == "pad_rows" else Lr))

    scale, shift = scale_shift(w, cfg)
    if mutate == "neighbour_block_bn":
        if len(scale) < 256:
            raise ValueError("neighbour_block_bn needs two filter blocks")
        scale, shift = scale.copy(), shift.copy()
        scale[128:256], shift[128:256] = scale[:128], shift[:128]
    if mutate == "abs_scale":
        scale = np.abs(scale)

    pads = list(pad_left(cfg))
    if mutate == "pad_shift":
        pads[0] += 1
    conv_pooled = []
    choff = 0
    for l, (k, F) in enumerate(zip(cfg.filter_lens, cfg.num_filters), 1):
        W = w[f"conv1d_{l}_W"][:, :, 0, :]
        if weights == "f16":
            W = W.astype(np.float16)
        Wk = W.astype(np.float64).transpose(2, 1, 0).reshape(k * 26, F)          # row j * 26 + channel
        # the one-hot windows of every output row: U[row, j * 26 + channel of residue t + j - pl]
        U = np.zeros((len(t), k * 26))
        for j in range(k - 1 if mutate == "drop_last_position" else k):
            r = t + j - pads[l - 1]
            ok = (r >= 0) & (r < Lr)
            ch = idx[sr[ok] + r[ok]]
            rows = np.nonzero(ok)[0]
            if mutate == "plane3_next_residue":
                keep = ch < 24
                rows, ch = rows[keep], ch[keep]
                r1 = r + 1
                ok1 = (r1 >= 0) & (r1 < Lr)
                ch1 = idx[sr[ok1] + r1[ok1]]
                hit = ch1 >= 24
                U[np.nonzero(ok1)[0][hit], j * 26 + ch1[hit]] = 1.0
            U[rows, j * 26 + ch] = 1.0
        P = np.empty((n, F))
        for f0 in range(0, F, _COLS):
            f1 = min(F, f0 + _COLS)
            y = U @ Wk[:, f0:f1]
            y = np.maximum(y * scale[choff + f0:choff + f1] + shift[choff + f0:choff + f1], 0.0)
            y[~pooled_rows] = 0.0                  # rows outside the pool never raise a max of ReLU outputs
            P[:, f0:f1] = np.maximum.reduceat(y, roff[:-1], axis=0)
        conv_pooled.append(P)
        choff += F
    pooled = np.concatenate(conv_pooled, axis=1)
    logits, scores = head(pooled, w, cfg.n_terms)
    return dict(lengths=L, conv_pooled=conv_pooled, pooled=pooled, logits=logits, scores=scores)
