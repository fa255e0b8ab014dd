"""ORACLE — TEST INFRASTRUCTURE ONLY (never imported by the product package).

Float64 restatement of upstream DeepFRI's GCN head (LSTM-LM -> embedding -> GraphConv x n -> sum-pool -> dense ->
FuncPredictor), written from the layer equations, not from the ONNX graph: it takes the weight dict of
`synth.make_weights(cfg, seed)` (exactly what `synth.write_gcn_model(path, cfg, seed)` serialises) and returns every stage, so
that a test can tell WHICH stage of an engine is off and by how much.

`deepfri_numpy` is the one-protein form (scores only).  `reference` runs a whole batch: the LSTM steps all proteins in
lockstep, one [B x H] . [H x 4H] product per time step over the proteins still running (a forward LSTM's output at step t
does not depend on later steps, so a protein that has ended simply leaves the product), and the X . W products of the
GraphConv layers run over all residues at once; only the L x L adjacency product is per protein.

`reference(..., mutate=<one of MUTANTS>)` computes the head with one defect of the kind the exact-fp32 engine's layout
(csrc/gcn_simt.cu) invites, for tests that show a bound would catch it.  The LSTM mutants act on every layer.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np

from cmap_oracle import seq2onehot


# defect -> what it does to the computation
MUTANTS = {
    "slice_edge": "unit 16 s + 15 takes its recurrent weights from the same unit of slice s + 1 (the next 16 units)",
    "gate_order": "the o and f gates trade places",
    "one_bias": "the LSTM bias is Wb alone, not Wb + Rb",
    "k_tail": "every GEMM (embedding, X.W, dense, labels) ignores its last K mod 16 inputs",
    "col_tail": "a GraphConv layer of 512 columns or more loses the columns past its last full 512-column pass",
    "row31": "row 32 k + 31 of every protein is left out of the aggregate (zero) and so of the pool",
    "pool_offset": "GraphConv layer l >= 2 adds its pooled slice at layer l - 1's offset",
    "depth_input": "LSTM layers 3 and 4 read layer 1's output",
    "second_chunk_stale_h": "a protein past the first 32 of its LSTM group gets h_{t-1} = 0",
}
LSTM_UNITS, LSTM_CHUNK = 16, 32        # units per CTA slice, proteins per chunk of a time step (csrc/gcn_simt.cu)


def lstm_groups(lengths, H, sm_count):
    """The exact-fp32 engine's LSTM schedule: proteins in length-descending stable order, dealt round-robin to
    min(sm_count / (H / 16), n) groups.  -> (n_groups, index of each protein within its group, in input order)."""
    n = len(lengths)
    n_groups = max(1, min(sm_count // (H // LSTM_UNITS), n))
    order = np.argsort(-np.asarray(lengths, np.int64), kind="stable")
    slot = np.empty(n, np.int64)
    slot[order] = np.arange(n) // n_groups
    return n_groups, slot


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


def lstm_batched(X: Sequence[np.ndarray], W, R, B, swap_of=False, one_bias=False, stale_h=None) -> List[np.ndarray]:
    """One ONNX LSTM layer (forward, zero state, gate order i, o, f, c) over a batch of sequences X[p] [L_p, in], in float64.
    Time step t multiplies the states of the proteins with L_p > t only: with the proteins ranked longest first, those are a
    prefix of the ranks, and the residues are laid out time-major (step t, then rank) so that each step reads and writes one
    contiguous block.  Mutants: `swap_of` trades the o and f gates, `one_bias` drops Rb, and proteins p with `stale_h[p]`
    see h_{t-1} = 0."""
    H = R.shape[-1]
    W, R = W[0].astype(np.float64), R[0].astype(np.float64)
    b = (B[0, :4 * H] + (0 if one_bias else B[0, 4 * H:])).astype(np.float64)
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
    keep = np.ones((len(X), 1)) if stale_h is None else (~np.asarray(stale_h, bool)[order]).astype(np.float64)[:, None]
    Wt, Rt = np.ascontiguousarray(W.T), np.ascontiguousarray(R.T)
    for t in range(Lmax):
        k = live[t]
        z = Xtm[start[t]:start[t + 1]] @ Wt + b + (h[:k] * keep[:k]) @ Rt
        i, o, f, g = _sigmoid(z[:, :H]), _sigmoid(z[:, H:2 * H]), _sigmoid(z[:, 2 * H:3 * H]), np.tanh(z[:, 3 * H:])
        if swap_of:
            o, f = f, o
        c[:k] = f * c[:k] + i * g
        h[:k] = o * np.tanh(c[:k])
        Y[start[t]:start[t + 1]] = h[:k]
    res = [None] * len(X)
    for r, p in enumerate(order):
        res[p] = Y[start[:Ls[r]] + r]
    return res


def _mutate_weights(w, cfg, mutate):
    """The weight dict with the weight-level defects applied (a copy where one is)."""
    if mutate == "slice_edge":
        H = cfg.lstm_hidden
        w = dict(w)
        src = np.arange(4 * H)
        for s in range(H // LSTM_UNITS):
            for g in range(4):
                src[g * H + LSTM_UNITS * s + 15] = g * H + (LSTM_UNITS * (s + 1) + 15) % H
        for l in range(1, cfg.lstm_layers + 1):
            w[f"lstm{l}_R"] = w[f"lstm{l}_R"][:, src]
    elif mutate == "k_tail":
        w = dict(w)
        keys = ["LM_embedding_W"] + [f"GraphConv_{l}_W" for l in range(1, len(cfg.gc_dims) + 1)] + ["dense_W", "labels_W"]
        for k in keys:
            K = w[k].shape[0]
            w[k] = w[k].copy()
            w[k][K - K % 16:] = 0
    return w


def reference(w: Dict[str, np.ndarray], cfg, seqs: Sequence[str], cmaps: Sequence[np.ndarray], mutate: Optional[str] = None,
              sm_count: int = 148) -> Dict[str, object]:
    """Every stage of the GCN head for a batch, in float64.  Per-residue stages are packed over the batch in input order
    (rows off[p]:off[p+1] belong to protein p, the layout of the engines' taps):
      hs[l] [T, H] (every LSTM layer), h1, h2 [T, H] (first and last LSTM layer), x0 [T, E], gc[l] [T, gc_dims[l]],
      d [T] (the degree normalisation 1 / (eps + sqrt(rowsum(A - diag A + I))));
    per protein: pooled [n, sum(gc_dims)] (every layer's sum over residues, concatenated as the engines lay it out),
      fc [n, F], logits [n, C, 2], scores [n, C].
    `mutate` names a defect of MUTANTS; `sm_count` (the SMs of the GPU) places the proteins in their LSTM groups for
    second_chunk_stale_h."""
    if mutate is not None and mutate not in MUTANTS:
        raise ValueError(f"unknown mutant {mutate!r}")
    w = _mutate_weights(w, cfg, mutate)
    n = len(seqs)
    lengths = np.array([len(s) for s in seqs], np.int64)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lengths, out=off[1:])
    S = [seq2onehot(s).astype(np.float64) for s in seqs]
    stale = lstm_groups(lengths, cfg.lstm_hidden, sm_count)[1] >= LSTM_CHUNK if mutate == "second_chunk_stale_h" and n else None
    hs, x, x1 = [], S, None
    for l in range(1, cfg.lstm_layers + 1):
        if mutate == "depth_input" and l >= 3:
            x = x1
        x = lstm_batched(x, w[f"lstm{l}_W"], w[f"lstm{l}_R"], w[f"lstm{l}_B"], swap_of=mutate == "gate_order",
                         one_bias=mutate == "one_bias", stale_h=stale)
        x1 = x if l == 1 else x1
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
        if mutate == "col_tail" and gd >= 512:
            x[:, gd // 512 * 512:] = 0
        if mutate == "row31":
            x[(np.arange(len(x)) - np.repeat(off[:-1], lengths)) % 32 == 31] = 0
        gc.append(x)
    cat = np.concatenate(gc, 1)
    pooled = np.stack([cat[off[p]:off[p + 1]].sum(0) for p in range(n)]) if n else np.zeros((0, cat.shape[1]))
    if mutate == "pool_offset":
        goff = np.concatenate([[0], np.cumsum(cfg.gc_dims)])
        moved = np.zeros_like(pooled)
        for l, gd in enumerate(cfg.gc_dims):
            at = goff[max(l - 1, 0)]
            moved[:, at:at + gd] += pooled[:, goff[l]:goff[l] + gd]
        pooled = moved
    fc = np.maximum(pooled @ w["dense_W"].astype(np.float64) + w["dense_b"], 0)
    logits = (fc @ w["labels_W"].astype(np.float64) + w["labels_b"]).reshape(n, -1, 2)
    e = np.exp(logits - logits.max(2, keepdims=True))
    scores = (e / e.sum(2, keepdims=True))[:, :, 0]
    return dict(off=off, hs=hs, h1=hs[0], h2=hs[-1], x0=x0, gc=gc, d=d, pooled=pooled, fc=fc, logits=logits, scores=scores)
