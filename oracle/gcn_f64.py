"""ORACLE — TEST INFRASTRUCTURE ONLY (never imported by the product package).

Float64 restatement of upstream DeepFRI's GCN head (LSTM-LM -> embedding -> GraphConv x n -> sum-pool -> dense ->
FuncPredictor), written from the layer equations, not from the ONNX graph: it takes the weight dict of
`synth.make_weights(cfg, seed)` (exactly what `synth.write_gcn_model(path, cfg, seed)` serialises) and returns every stage, so
that a test can tell WHICH stage of an engine is off and by how much.

`deepfri_numpy` is the one-protein form (scores only).  `reference` runs a whole batch: the LSTM steps all proteins in
lockstep, one [B x H] . [H x 4H] product per time step over the proteins still running (a forward LSTM's output at step t
does not depend on later steps, so a protein that has ended simply leaves the product), and the X . W products of the
GraphConv layers run over all residues at once; only the L x L adjacency product is per protein.
"""
from __future__ import annotations

from typing import Dict, List, Sequence

import numpy as np

from cmap_oracle import seq2onehot


def _sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def _act(z, cfg):
    return np.where(z > 0, z, np.expm1(np.minimum(z, 0))) if cfg.gc_activation == "Elu" else np.maximum(z, 0)


def deepfri_numpy(w, cfg, seq, cmap):
    """Independent float64 restatement of upstream DeepFRI's equations for one protein (not the ONNX interpreter)."""
    S = seq2onehot(seq).astype(np.float64)
    H = cfg.lstm_hidden

    def lstm(X, W, R, B):
        W, R = W[0].astype(np.float64), R[0].astype(np.float64)
        b = (B[0, :4 * H] + B[0, 4 * H:]).astype(np.float64)
        h = np.zeros(H); c = np.zeros(H); out = []
        for x in X:
            z = W @ x + R @ h + b
            i, o, f, g = _sigmoid(z[:H]), _sigmoid(z[H:2 * H]), _sigmoid(z[2 * H:3 * H]), np.tanh(z[3 * H:])
            c = f * c + i * g
            h = o * np.tanh(c)
            out.append(h)
        return np.array(out)
    h = S
    for l in range(1, cfg.lstm_layers + 1):
        h = lstm(h, w[f"lstm{l}_W"], w[f"lstm{l}_R"], w[f"lstm{l}_B"])
    x = np.maximum(h @ w["LM_embedding_W"] + w["LM_embedding_b"] + S @ w["AA_embedding_W"], 0)
    A = cmap.astype(np.float64)
    A = A - np.diag(np.diag(A)) + np.eye(len(A))
    d = 1.0 / (cfg.eps + np.sqrt(A.sum(1)))
    An = d[:, None] * A * d[None, :]
    outs = []
    for l in range(1, len(cfg.gc_dims) + 1):
        z = (An @ x) @ w[f"GraphConv_{l}_W"]
        if cfg.gc_bias:
            z = z + w[f"GraphConv_{l}_b"]
        x = _act(z, cfg)
        outs.append(x)
    p = np.concatenate(outs, 1).sum(0)
    f = np.maximum(p @ w["dense_W"] + w["dense_b"], 0)
    o = (f @ w["labels_W"] + w["labels_b"]).reshape(-1, 2)
    e = np.exp(o - o.max(1, keepdims=True))
    return (e / e.sum(1, keepdims=True))[:, 0]


def lstm_batched(X: Sequence[np.ndarray], W, R, B) -> List[np.ndarray]:
    """One ONNX LSTM layer (forward, zero state, gate order i, o, f, c) over a batch of sequences X[p] [L_p, in], in float64.
    Time step t multiplies the states of the proteins with L_p > t only: with the proteins ranked longest first, those are a
    prefix of the ranks, and the residues are laid out time-major (step t, then rank) so that each step reads and writes one
    contiguous block."""
    H = R.shape[-1]
    W, R = W[0].astype(np.float64), R[0].astype(np.float64)
    b = (B[0, :4 * H] + B[0, 4 * H:]).astype(np.float64)
    lengths = np.array([len(x) for x in X], np.int64)
    order = np.argsort(-lengths, kind="stable")
    Ls = lengths[order]
    Lmax = int(Ls[0]) if len(Ls) else 0
    live = np.searchsorted(-Ls, -np.arange(Lmax), side="left")       # proteins still running at step t
    start = np.zeros(Lmax + 1, np.int64)
    np.cumsum(live, out=start[1:])
    Xtm = np.zeros((int(start[-1]), W.shape[1]))
    for r, p in enumerate(order):
        Xtm[start[:Ls[r]] + r] = X[p]
    Y = np.zeros((len(Xtm), H))
    h = np.zeros((len(X), H)); c = np.zeros((len(X), H))
    Wt, Rt = np.ascontiguousarray(W.T), np.ascontiguousarray(R.T)
    for t in range(Lmax):
        k = live[t]
        z = Xtm[start[t]:start[t + 1]] @ Wt + b + h[:k] @ Rt
        i, o, f, g = _sigmoid(z[:, :H]), _sigmoid(z[:, H:2 * H]), _sigmoid(z[:, 2 * H:3 * H]), np.tanh(z[:, 3 * H:])
        c[:k] = f * c[:k] + i * g
        h[:k] = o * np.tanh(c[:k])
        Y[start[t]:start[t + 1]] = h[:k]
    res = [None] * len(X)
    for r, p in enumerate(order):
        res[p] = Y[start[:Ls[r]] + r]
    return res


def reference(w: Dict[str, np.ndarray], cfg, seqs: Sequence[str], cmaps: Sequence[np.ndarray]) -> Dict[str, object]:
    """Every stage of the GCN head for a batch, in float64.  Per-residue stages are packed over the batch in input order
    (rows off[p]:off[p+1] belong to protein p, the layout of the engines' taps):
      h1, h2 [T, H] (first and last LSTM layer), x0 [T, E], gc[l] [T, gc_dims[l]],
      d [T] (the degree normalisation 1 / (eps + sqrt(rowsum(A - diag A + I))));
    per protein: pooled [n, sum(gc_dims)] (every layer's sum over residues, concatenated as the engines lay it out),
      fc [n, F], logits [n, C, 2], scores [n, C]."""
    n = len(seqs)
    lengths = np.array([len(s) for s in seqs], np.int64)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lengths, out=off[1:])
    S = [seq2onehot(s).astype(np.float64) for s in seqs]
    hs, x = [], S
    for l in range(1, cfg.lstm_layers + 1):
        x = lstm_batched(x, w[f"lstm{l}_W"], w[f"lstm{l}_R"], w[f"lstm{l}_B"])
        hs.append(np.concatenate(x) if n else np.zeros((0, cfg.lstm_hidden)))
    Sp = np.concatenate(S) if n else np.zeros((0, cfg.n_channels))
    x0 = np.maximum(hs[-1] @ w["LM_embedding_W"].astype(np.float64) + w["LM_embedding_b"] + Sp @ w["AA_embedding_W"].astype(np.float64), 0)
    d = np.zeros(int(off[-1]))
    A_hat = []
    for p in range(n):
        A = np.asarray(cmaps[p], np.float64)
        if A.shape != (lengths[p], lengths[p]):
            raise ValueError(f"protein {p}: contact map {A.shape} does not match its length {lengths[p]}")
        A = A - np.diag(np.diag(A)) + np.eye(len(A))
        d[off[p]:off[p + 1]] = 1.0 / (cfg.eps + np.sqrt(A.sum(1)))
        A_hat.append(A)
    gc, x = [], x0
    for l, gd in enumerate(cfg.gc_dims, 1):
        y = d[:, None] * (x @ w[f"GraphConv_{l}_W"].astype(np.float64))          # (D A D) X W = D (A (D X W))
        z = np.empty((len(y), gd))
        for p in range(n):
            s = slice(off[p], off[p + 1])
            z[s] = d[s, None] * (A_hat[p] @ y[s])
        if cfg.gc_bias:
            z += w[f"GraphConv_{l}_b"]
        x = _act(z, cfg)
        gc.append(x)
    cat = np.concatenate(gc, 1)
    pooled = np.stack([cat[off[p]:off[p + 1]].sum(0) for p in range(n)]) if n else np.zeros((0, cat.shape[1]))
    fc = np.maximum(pooled @ w["dense_W"].astype(np.float64) + w["dense_b"], 0)
    logits = (fc @ w["labels_W"].astype(np.float64) + w["labels_b"]).reshape(n, -1, 2)
    e = np.exp(logits - logits.max(2, keepdims=True))
    scores = (e / e.sum(2, keepdims=True))[:, :, 0]
    return dict(off=off, h1=hs[0], h2=hs[-1], x0=x0, gc=gc, d=d, pooled=pooled, fc=fc, logits=logits, scores=scores)
