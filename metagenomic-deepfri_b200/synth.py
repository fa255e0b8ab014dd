"""Synthetic models and workloads (SURVEY.md §8d).

Nothing here is on the product path: it writes random-init DeepFRI GCN heads *in the
reference's ONNX layout* (the file `mDeepFRI.predict.Predictor` hands to onnxruntime,
`predict.pyx:62-73`; model family `DeepFRI-MERGED_GraphConv_gcd_512-512-512_fcd_1024_ca_10.0_*`,
`mDeepFRI/__init__.py:73`) and generates seeded proteins / structures / alignments for the
BASELINE.json configs.  The real `.onnx` files are not redistributable offline, so the graph
below restates upstream DeepFRI (LSTM-LM -> GraphConv x3 -> sum-pool -> dense -> FuncPredictor)
with standard ONNX ops the way tf2onnx lowers a Keras model (Transpose/LSTM/Squeeze,
MatMul/Add, Elu, ReduceSum, Reshape, Softmax).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import onnx_lite as ox

AA20 = "ACDEFGHIKLMNPQRSTVWY"
# head sizes of the v1.0 "MERGED" models (SURVEY.md §3.3)
HEAD_SIZES = {"mf": 489, "bp": 1943, "cc": 320, "ec": 538}


@dataclass
class GCNConfig:
    n_channels: int = 26
    lstm_hidden: int = 512          # LSTM-LM hidden size H (every layer)
    lstm_layers: int = 2            # LSTM-LM depth (upstream DeepFRI: 2)
    lm_dim: int = 1024              # embedding width E
    gc_dims: Tuple[int, ...] = (512, 512, 512)
    fc_dim: int = 1024
    n_terms: int = 489              # C
    gc_activation: str = "Elu"      # upstream GraphConv uses elu; north-star text says ReLU
    gc_bias: bool = False
    eps: float = 1e-6
    logit_scale: float = 0.0125      # multiplies the FuncPredictor dense so scores are not saturated


def _uniform(rng, a, shape):
    return rng.uniform(-a, a, size=shape).astype(np.float32)


def make_weights(cfg: GCNConfig, seed: int = 1234, lm_seed: int = 99) -> Dict[str, np.ndarray]:
    """Random-init weights with gains chosen so that activations are O(0.1-1) like a trained
    network (plain Glorot leaves the LSTM-LM output ~1e-2 and would hide LSTM / GraphConv
    arithmetic errors from the parity tests).  LSTM biases 0 with forget gate 1 (Keras).

    The LSTM-LM uses its own seed so that every head shares byte-identical LM weights,
    as upstream freezes the language model (SURVEY.md §3.3)."""
    H, E, I = cfg.lstm_hidden, cfg.lm_dim, cfg.n_channels
    lm = np.random.default_rng(lm_seed)
    rng = np.random.default_rng(seed)
    w: Dict[str, np.ndarray] = {}
    rec = np.sqrt(3.0 / H) * 1.5
    for l in range(1, cfg.lstm_layers + 1):
        inp = I if l == 1 else H
        # ONNX LSTM layout: W[1,4H,in], R[1,4H,H], B[1,8H]; gate order i,o,f,c
        w[f"lstm{l}_W"] = _uniform(lm, 1.5 if l == 1 else rec * 2.0, (1, 4 * H, inp))
        w[f"lstm{l}_R"] = _uniform(lm, rec, (1, 4 * H, H))
        b = _uniform(lm, 0.1, (1, 8 * H))
        b[0, 2 * H:3 * H] += 1.0     # forget-gate bias (input half)
        w[f"lstm{l}_B"] = b
    w["AA_embedding_W"] = _uniform(rng, 0.5, (I, E))
    w["LM_embedding_W"] = _uniform(rng, np.sqrt(6.0 / H), (H, E))
    w["LM_embedding_b"] = _uniform(rng, 0.1, (E,))
    prev = E
    for l, g in enumerate(cfg.gc_dims, 1):
        w[f"GraphConv_{l}_W"] = _uniform(rng, np.sqrt(6.0 / prev) * 1.4, (prev, g))
        if cfg.gc_bias:
            w[f"GraphConv_{l}_b"] = _uniform(rng, 0.1, (g,))
        prev = g
    G = int(sum(cfg.gc_dims))
    w["dense_W"] = _uniform(rng, np.sqrt(6.0 / (G + cfg.fc_dim)), (G, cfg.fc_dim))
    w["dense_b"] = _uniform(rng, 0.1, (cfg.fc_dim,))
    w["labels_W"] = _uniform(rng, np.sqrt(6.0 / (cfg.fc_dim + 2 * cfg.n_terms)) * cfg.logit_scale,
                             (cfg.fc_dim, 2 * cfg.n_terms))
    w["labels_b"] = _uniform(rng, 1.0, (2 * cfg.n_terms,))
    return w


def build_gcn_model(cfg: GCNConfig, weights: Optional[Dict[str, np.ndarray]] = None,
                    seed: int = 1234, style: str = "compact") -> ox.Model:
    """DeepFRI GCN head as an ONNX graph. Inputs are ordered (cmap, seq) as the reference
    feeds them (`predict.pyx:87-90`); output is [1, C, 2] with the score in channel 0
    (`predict.pyx:100`).

    `style="compact"`: the adjacency is normalised once (D.A.D as two broadcast Muls) and shared by the layers.
    `style="tf2onnx"`: closer to what tf2onnx makes of upstream's Keras layers - every GraphConv layer carries its own
    copy of `GraphConv._normalize` with D_hat an explicit diagonal MATRIX and `matmul(matmul(D_hat, A_hat), D_hat)`
    (three data-dependent MatMuls per layer), `eps + sqrt(.)` with the constant on the left, and the LSTM nodes carry an
    empty sequence_lens, constant-zero initial_h / initial_c and the Y_h / Y_c outputs.  Same function, same weights."""
    if style not in ("compact", "tf2onnx"):
        raise ValueError(style)
    w = dict(weights) if weights is not None else make_weights(cfg, seed)
    g = ox.Graph(name="DeepFRI_GraphConv")
    g.inputs = [ox.ValueInfo("cmap", ox.FLOAT, ("unk__b", "unk__l", "unk__l")),
                ox.ValueInfo("seq", ox.FLOAT, ("unk__b", "unk__l", cfg.n_channels))]
    g.outputs = [ox.ValueInfo("labels", ox.FLOAT, ("unk__b", cfg.n_terms, 2))]
    init = g.initializers
    N = g.nodes
    for k, v in w.items():
        init[k] = v
    init["const_axes_0"] = np.array([0], np.int64)
    init["const_axes_1"] = np.array([1], np.int64)
    init["const_axes_2"] = np.array([2], np.int64)
    init["const_one"] = np.array(1.0, np.float32)
    init["const_eps"] = np.array(cfg.eps, np.float32)
    init["const_out_shape"] = np.array([-1, cfg.n_terms, 2], np.int64)

    def add(op, ins, outs, **attrs):
        N.append(ox.Node(op, list(ins), list(outs), name=f"{op}__{len(N)}", attrs=attrs))
        return outs[0]

    # ---- LSTM language model (tf2onnx: Transpose -> LSTM -> Squeeze, time-major)
    H = cfg.lstm_hidden
    x = add("Transpose", ["seq"], ["lm/seq_tm"], perm=[1, 0, 2])
    if style == "tf2onnx":
        init["lm/zero_state"] = np.zeros((1, 1, H), np.float32)
    for l in range(1, cfg.lstm_layers + 1):
        if style == "tf2onnx":
            y = add("LSTM", [x, f"lstm{l}_W", f"lstm{l}_R", f"lstm{l}_B", "", "lm/zero_state", "lm/zero_state"],
                    [f"lm/LSTM{l}_Y", f"lm/LSTM{l}_Yh", f"lm/LSTM{l}_Yc"], hidden_size=H, direction="forward")
        else:
            y = add("LSTM", [x, f"lstm{l}_W", f"lstm{l}_R", f"lstm{l}_B"],
                    [f"lm/LSTM{l}_Y"], hidden_size=H, direction="forward")
        x = add("Squeeze", [y, "const_axes_1"], [f"lm/LSTM{l}_out"])
    lm_out = add("Transpose", [x], [f"lm/LSTM{cfg.lstm_layers}_bm"], perm=[1, 0, 2])
    x_lm = add("MatMul", [lm_out, "LM_embedding_W"], ["LM_embedding/MatMul"])
    x_lm = add("Add", [x_lm, "LM_embedding_b"], ["LM_embedding/BiasAdd"])
    x_aa = add("MatMul", ["seq", "AA_embedding_W"], ["AA_embedding/MatMul"])
    x = add("Add", [x_lm, x_aa], ["Embedding/add"])
    x = add("Relu", [x], ["activation/Relu"])

    # ---- adjacency normalisation (GraphConv._normalize upstream)
    def normalize(pfx: str, matrix_form: bool) -> str:
        a2 = add("Squeeze", ["cmap", "const_axes_0"], [pfx + "A2d"])
        eye = add("EyeLike", [a2], [pfx + "eye2d"])
        eye = add("Unsqueeze", [eye, "const_axes_0"], [pfx + "eye"])
        dg = add("Mul", ["cmap", eye], [pfx + "diagA"])
        a0 = add("Sub", ["cmap", dg], [pfx + "A_nodiag"])
        ah = add("Add", [a0, eye], [pfx + "A_hat"])
        rs = add("ReduceSum", [ah, "const_axes_2"], [pfx + "rowsum"], keepdims=0)
        sq = add("Sqrt", [rs], [pfx + "sqrt"])
        dn = add("Add", ["const_eps", sq] if matrix_form else [sq, "const_eps"], [pfx + "denom"])
        d = add("Div", ["const_one", dn], [pfx + "d"])
        dc = add("Unsqueeze", [d, "const_axes_2"], [pfx + "d_col"])
        if matrix_form:
            dm = add("Mul", [dc, eye], [pfx + "D_hat"])                       # tf.linalg.diag(d)
            da = add("MatMul", [dm, ah], [pfx + "DA"])
            return add("MatMul", [da, dm], [pfx + "DAD"])
        dr = add("Unsqueeze", [d, "const_axes_1"], [pfx + "d_row"])
        da = add("Mul", [dc, ah], [pfx + "DA"])
        return add("Mul", [da, dr], [pfx + "DAD"])

    an = normalize("norm/", False) if style == "compact" else None

    # ---- GraphConv stack: act((A_n . X) . W [+ b])
    outs = []
    for l, gdim in enumerate(cfg.gc_dims, 1):
        if style == "tf2onnx":
            an = normalize(f"GraphConv_{l}/norm/", True)
        t = add("MatMul", [an, x], [f"GraphConv_{l}/batch_dot"])
        t = add("MatMul", [t, f"GraphConv_{l}_W"], [f"GraphConv_{l}/MatMul"])
        if cfg.gc_bias:
            t = add("Add", [t, f"GraphConv_{l}_b"], [f"GraphConv_{l}/BiasAdd"])
        if cfg.gc_activation == "Elu":
            x = add("Elu", [t], [f"GraphConv_{l}/Elu"], alpha=1.0)
        else:
            x = add(cfg.gc_activation, [t], [f"GraphConv_{l}/{cfg.gc_activation}"])
        outs.append(x)
    cat = add("Concat", outs, ["GCNN_concatenate/concat"], axis=2) if len(outs) > 1 else outs[0]
    pooled = add("ReduceSum", [cat, "const_axes_1"], ["SumPooling/Sum"], keepdims=0)
    h = add("MatMul", [pooled, "dense_W"], ["dense/MatMul"])
    h = add("Add", [h, "dense_b"], ["dense/BiasAdd"])
    h = add("Relu", [h], ["dense/Relu"])
    o = add("MatMul", [h, "labels_W"], ["labels/dense/MatMul"])
    o = add("Add", [o, "labels_b"], ["labels/dense/BiasAdd"])
    o = add("Reshape", [o, "const_out_shape"], ["labels/reshape"])
    add("Softmax", [o], ["labels"], axis=-1)
    return ox.Model(g, ir_version=8, opset=15, producer_name="mdf-b200-synth",
                    producer_version="1")


def write_gcn_model(path: str, cfg: GCNConfig, seed: int = 1234, style: str = "compact") -> None:
    ox.save(build_gcn_model(cfg, seed=seed, style=style), path)


# ----------------------------------------------------------------------------- sequence-only DeepCNN heads
@dataclass
class CNNConfig:
    """Upstream DeepFRI `DeepCNN` (the `DeepCNN-MERGED_*` models, `mDeepFRI/__init__.py:68`): parallel Conv1D layers over
    the one-hot sequence, concatenated, BatchNormalization, ReLU, global max-pool, FuncPredictor.  Defaults = the trained
    models' 16 x 512 filters of widths 8..128."""
    n_channels: int = 26
    filter_lens: Tuple[int, ...] = tuple(range(8, 129, 8))
    num_filters: Tuple[int, ...] = (512,) * 16
    n_terms: int = 489
    bn_epsilon: float = 1e-3          # Keras BatchNormalization default
    logit_scale: float = 0.15
    pad_left: Optional[Tuple[int, ...]] = None   # zeros before position 0 per conv; None: Keras 'same', (k - 1) // 2


def make_cnn_weights(cfg: CNNConfig, seed: int = 4321) -> Dict[str, np.ndarray]:
    rng = np.random.default_rng(seed)
    w: Dict[str, np.ndarray] = {}
    for l, (k, f) in enumerate(zip(cfg.filter_lens, cfg.num_filters), 1):
        # ONNX Conv weight [F, C, 1, k] (tf2onnx lowers Keras Conv1D to a Conv over [N, C, 1, L]); one-hot input: a window sums
        # k weights, so a gain of ~1/sqrt(k) keeps the pre-activations O(1)
        w[f"conv1d_{l}_W"] = _uniform(rng, np.sqrt(3.0 / k), (f, cfg.n_channels, 1, k))
        w[f"conv1d_{l}_b"] = _uniform(rng, 0.1, (f,))
    tot = int(sum(cfg.num_filters))
    w["bn_gamma"] = rng.uniform(0.5, 1.5, tot).astype(np.float32)
    w["bn_beta"] = _uniform(rng, 0.3, (tot,))
    w["bn_mean"] = _uniform(rng, 0.3, (tot,))
    w["bn_var"] = rng.uniform(0.5, 1.5, tot).astype(np.float32)
    w["labels_W"] = _uniform(rng, np.sqrt(6.0 / (tot + 2 * cfg.n_terms)) * cfg.logit_scale, (tot, 2 * cfg.n_terms))
    w["labels_b"] = _uniform(rng, 1.0, (2 * cfg.n_terms,))
    return w


def build_cnn_model(cfg: CNNConfig, weights: Optional[Dict[str, np.ndarray]] = None, seed: int = 4321) -> ox.Model:
    """DeepCNN head as an ONNX graph in tf2onnx style: one input `seq` [b, L, 26] (the reference feeds it alone,
    `predict.pyx:91-95`), channels-first Conv nodes with explicit pads (cfg.pad_left before, default TF 'same' (k-1)//2,
    and the rest of k - 1 after),
    Concat, BatchNormalization, Relu, ReduceMax over residues, MatMul/Add, Reshape, Softmax -> [1, C, 2]."""
    w = dict(weights) if weights is not None else make_cnn_weights(cfg, seed)
    g = ox.Graph(name="DeepCNN")
    g.inputs = [ox.ValueInfo("seq", ox.FLOAT, ("unk__b", "unk__l", cfg.n_channels))]
    g.outputs = [ox.ValueInfo("labels", ox.FLOAT, ("unk__b", cfg.n_terms, 2))]
    init, N = g.initializers, g.nodes
    for k, v in w.items():
        init[k] = v
    init["const_axes_2"] = np.array([2], np.int64)
    init["const_out_shape"] = np.array([-1, cfg.n_terms, 2], np.int64)

    def add(op, ins, outs, **attrs):
        N.append(ox.Node(op, list(ins), list(outs), name=f"{op}__{len(N)}", attrs=attrs))
        return outs[0]

    x = add("Transpose", ["seq"], ["seq_cf"], perm=[0, 2, 1])                 # [b, 26, L]
    x = add("Unsqueeze", [x, "const_axes_2"], ["seq_cf4"])                    # [b, 26, 1, L]
    outs = []
    for l, k in enumerate(cfg.filter_lens, 1):
        pl = cfg.pad_left[l - 1] if cfg.pad_left is not None else (k - 1) // 2
        y = add("Conv", [x, f"conv1d_{l}_W", f"conv1d_{l}_b"], [f"conv1d_{l}/Conv2D"], kernel_shape=[1, k], strides=[1, 1],
                dilations=[1, 1], group=1, pads=[0, pl, 0, k - 1 - pl])
        outs.append(add("Squeeze", [y, "const_axes_2"], [f"conv1d_{l}/Squeeze"]))   # [b, F, L]
    cat = add("Concat", outs, ["concatenate/concat"], axis=1) if len(outs) > 1 else outs[0]
    bn = add("BatchNormalization", [cat, "bn_gamma", "bn_beta", "bn_mean", "bn_var"], ["batch_normalization/bn"],
             epsilon=float(cfg.bn_epsilon), momentum=0.99)
    r = add("Relu", [bn], ["CAM_layer/Relu"])
    p = add("ReduceMax", [r], ["global_max_pooling1d/Max"], axes=[2], keepdims=0)   # [b, sum F]
    o = add("MatMul", [p, "labels_W"], ["labels/dense/MatMul"])
    o = add("Add", [o, "labels_b"], ["labels/dense/BiasAdd"])
    o = add("Reshape", [o, "const_out_shape"], ["labels/reshape"])
    add("Softmax", [o], ["labels"], axis=-1)
    return ox.Model(g, ir_version=8, opset=15, producer_name="mdf-b200-synth", producer_version="1")


def write_cnn_model(path: str, cfg: CNNConfig, seed: int = 4321) -> None:
    ox.save(build_cnn_model(cfg, seed=seed), path)


# ----------------------------------------------------------------------------- workloads
def random_sequences(rng: np.random.Generator, lengths: Sequence[int]) -> List[str]:
    """Uniform over the 20 standard residues."""
    table = np.frombuffer(AA20.encode(), dtype=np.uint8)
    flat = table[rng.integers(0, 20, size=int(np.sum(lengths)))]
    out, p = [], 0
    for L in lengths:
        out.append(flat[p:p + L].tobytes().decode())
        p += L
    return out


def random_walk_coords(rng: np.random.Generator, lengths: Sequence[int],
                       step: float = 3.8, pull: float = 0.0, persist: float = 0.5) -> List[np.ndarray]:
    """Calpha random walks: 3.8 A steps, direction = random + `persist` x previous direction
    (+ optional weak pull toward the running centroid), rounded to 3 decimals (PDB
    precision).  Defaults give protein-like contact density: ~13-21 contacts per residue at
    10 A and ~5-8 at 6 A.  Vectorised over proteins, sequential over residues."""
    lengths = np.asarray(lengths, dtype=np.int64)
    n, Lmax = len(lengths), int(lengths.max()) if len(lengths) else 0
    pos = np.zeros((n, 3), np.float64)
    csum = np.zeros((n, 3), np.float64)
    vprev = np.zeros((n, 3), np.float64)
    out = np.zeros((Lmax, n, 3), np.float32)
    for t in range(Lmax):
        if t:
            v = rng.standard_normal((n, 3))
            v /= np.linalg.norm(v, axis=1, keepdims=True) + 1e-12
            v = v + persist * vprev + pull * (csum / t - pos)
            v /= np.linalg.norm(v, axis=1, keepdims=True) + 1e-12
            pos = pos + step * v
            vprev = v
        csum += pos
        out[t] = np.round(pos, 3).astype(np.float32)
    return [np.ascontiguousarray(out[:L, i]) for i, L in enumerate(lengths)]


def markov_alignments(rng: np.random.Generator, queries: Sequence[str],
                      p_open: float = 0.02, p_ext: float = 0.5, p_match: float = 0.6
                      ) -> Tuple[List[str], List[str], List[str]]:
    """MMseqs2/PyOpal-style pairwise alignments from a 3-state Markov chain over
    {M, I, D}.  `I` puts '-' in the query, `D` puts '-' in the target — the dialect of
    `mDeepFRI.alignment.insert_gaps` (`alignment.py:38-62`).  Returns
    (gapped_query, gapped_target, target_sequence)."""
    gq_all, gt_all, tgt_all = [], [], []
    aa = np.frombuffer(AA20.encode(), dtype=np.uint8)
    for q in queries:
        Lq = len(q)
        qb = np.frombuffer(q.encode(), dtype=np.uint8)
        # run-length form of the chain: M-run, gap-run (I or D), M-run, ...; more runs than
        # needed are drawn, then the columns are cut where the query is consumed
        k = int(Lq * 2 * p_open * 1.5) + 8
        m_len = rng.geometric(2 * p_open, size=k)
        if rng.random() < 0.05:
            m_len[0] = 0                                   # leading gap
        g_len = rng.geometric(1.0 - p_ext, size=k)
        g_typ = rng.integers(1, 3, size=k).astype(np.int8)  # 1=I 2=D
        runs_state = np.empty(2 * k, np.int8)
        runs_state[0::2] = 0
        runs_state[1::2] = g_typ
        runs_len = np.empty(2 * k, np.int64)
        runs_len[0::2] = m_len
        runs_len[1::2] = g_len
        state = np.repeat(runs_state, runs_len)            # 0=M 1=I 2=D per column
        consumes_q = state != 1
        cq = np.cumsum(consumes_q)
        if cq[-1] < Lq:                                    # (rare) not enough columns: pad with M
            state = np.concatenate([state, np.zeros(Lq - cq[-1], np.int8)])
            consumes_q = state != 1
            cq = np.cumsum(consumes_q)
        end = int(np.searchsorted(cq, Lq)) + 1
        if rng.random() < 0.05:                            # trailing query gap
            state = np.concatenate([state[:end], np.ones(int(rng.integers(1, 4)), np.int8)])
            end = len(state)
        state = state[:end]
        consumes_q = state != 1
        assert int(consumes_q.sum()) == Lq
        qi = np.cumsum(consumes_q) - 1
        gq = np.where(consumes_q, qb[np.clip(qi, 0, Lq - 1)], ord("-")).astype(np.uint8)
        rnd = aa[rng.integers(0, 20, size=end)]
        keep = rng.random(end) < p_match
        tcol = np.where((state == 0) & keep, gq, rnd)
        gt = np.where(state == 2, ord("-"), tcol).astype(np.uint8)
        gq_all.append(gq.tobytes().decode())
        gt_all.append(gt.tobytes().decode())
        tgt_all.append(gt[gt != ord("-")].tobytes().decode())
    return gq_all, gt_all, tgt_all


@dataclass
class Workload:
    """One batch of the hot path's inputs (what `pipeline.py:476-481` + `:301-319` consume)."""
    query_seqs: List[str]
    gapped_query: List[str]
    gapped_target: List[str]
    coords: List[np.ndarray]          # float32 [Lt, 3] per target structure
    threshold: float = 10.0
    generated_contacts: int = 2
    name: str = ""

    def __len__(self):
        return len(self.query_seqs)


def make_workload(n: int, lmin: int, lmax: int, seed: int, *, gapped: bool = True,
                  threshold: float = 10.0, generated_contacts: int = 2,
                  dist: str = "uniform", name: str = "") -> Workload:
    rng = np.random.default_rng(seed)
    if dist == "uniform":
        lengths = rng.integers(lmin, lmax + 1, size=n)
    elif dist == "lognormal":       # metagenomic length distribution, SURVEY.md §8d config 3
        lengths = np.clip(np.exp(rng.normal(np.log(250.0), 0.6, size=n)), lmin, lmax).astype(np.int64)
    else:
        raise ValueError(dist)
    seqs = random_sequences(rng, lengths)
    if gapped:
        gq, gt, tgt = markov_alignments(rng, seqs)
    else:
        gq, gt, tgt = list(seqs), list(seqs), list(seqs)
    coords = random_walk_coords(rng, [len(t) for t in tgt])
    return Workload(seqs, gq, gt, coords, threshold, generated_contacts,
                    name or f"n{n}_L{lmin}-{lmax}_{dist}_seed{seed}")


# ----------------------------------------------------------------------------- keyed generator (the sharded 1M-protein job)
# Protein i of a job is a pure function of (seed, i): any rank can generate exactly its own shard of BASELINE configs[4] without
# generating (or receiving) the rest, whatever the number of ranks.  Counter-based: every random number is a splitmix64 hash of
# (seed, protein, position, channel).  Same model as make_workload: L ~ LogNormal(median 250, sigma 0.6) clipped, uniform
# residues, Markov-gapped alignments (gap open 0.02 + 0.02, extension 0.5, 5 % leading / trailing gaps, 60 % identity),
# C-alpha random walks with 3.8 A steps and 0.5 direction persistence, coordinates rounded to 3 decimals.
_G = np.uint64(0x9E3779B97F4A7C15)
_M1, _M2 = np.uint64(0xBF58476D1CE4E5B9), np.uint64(0x94D049BB133111EB)
_K1, _K2 = np.uint64(0xD6E8FEB86659FD93), np.uint64(0xA24BAED4963EE407)


def _mix64(x: np.ndarray) -> np.ndarray:
    x = (x ^ (x >> np.uint64(30))) * _M1
    x = (x ^ (x >> np.uint64(27))) * _M2
    return x ^ (x >> np.uint64(31))


def _hash(base: np.ndarray, t, c: int) -> np.ndarray:
    """base = per-protein key (uint64), t = position (scalar or array), c = channel."""
    with np.errstate(over="ignore"):
        return _mix64(base + np.uint64(t) * _K1 + np.uint64(c) * _K2) if np.isscalar(t) else \
            _mix64(base + t.astype(np.uint64) * _K1 + np.uint64(c) * _K2)


def _u01(h: np.ndarray) -> np.ndarray:
    return ((h >> np.uint64(11)).astype(np.float64) + 0.5) * (2.0 ** -53)


def _protein_keys(ids: np.ndarray, seed: int) -> np.ndarray:
    with np.errstate(over="ignore"):
        return _mix64(np.asarray(ids, np.uint64) * _G + np.uint64(seed) * _K2 + _K1)


def keyed_lengths(ids: Sequence[int], seed: int, lmin: int = 50, lmax: int = 1000) -> np.ndarray:
    """Query lengths of the proteins `ids` of job `seed` (cheap: the LPT partition needs all of them on every rank)."""
    k = _protein_keys(np.asarray(ids, np.int64), seed)
    z = np.sqrt(-2.0 * np.log(_u01(_hash(k, 0, 101)))) * np.cos(2.0 * np.pi * _u01(_hash(k, 0, 102)))
    return np.clip(np.exp(np.log(250.0) + 0.6 * z), lmin, lmax).astype(np.int64)


def keyed_workload(ids: Sequence[int], seed: int, lmin: int = 50, lmax: int = 1000, threshold: float = 10.0,
                   generated_contacts: int = 2, name: str = "") -> Workload:
    ids = np.asarray(ids, np.int64)
    n = len(ids)
    if n == 0:
        return Workload([], [], [], [], threshold, generated_contacts, name)
    key = _protein_keys(ids, seed)
    L = keyed_lengths(ids, seed, lmin, lmax)
    aa = np.frombuffer(AA20.encode(), np.uint8)
    # ---- alignment columns: state 0 = M, 1 = I ('-' in the query), 2 = D ('-' in the target); one column per step for all proteins
    cap = int(L.max() * 1.25) + 64
    state = np.full((n, cap), 3, np.int8)                  # 3 = past the end
    qpos = np.zeros(n, np.int64)                           # query residues consumed so far
    cur = np.where(_u01(_hash(key, 0, 1)) < 0.05, np.where(_hash(key, 0, 2) & np.uint64(1), 1, 2), 0).astype(np.int8)   # leading gap
    ncols = np.zeros(n, np.int64)
    alive = np.arange(n)
    for col in range(cap):
        if alive.size == 0:
            break
        k, c = key[alive], cur[alive]
        state[alive, col] = c
        qpos[alive] += c != 1
        ncols[alive] = col + 1
        u = _u01(_hash(k, col, 3))
        gap_type = np.where(_hash(k, col, 4) & np.uint64(1), 1, 2).astype(np.int8)
        nxt = np.where(c == 0, np.where(u < 0.04, gap_type, 0), np.where(u < 0.5, c, 0)).astype(np.int8)
        cur[alive] = nxt
        done = qpos[alive] >= L[alive]
        alive = alive[~done]
    if alive.size:
        raise RuntimeError("keyed_workload: alignment did not terminate (raise the column capacity)")
    # trailing query gap (5 %): 1-3 extra I columns
    trail = np.where(_u01(_hash(key, 0, 5)) < 0.05, 1 + (_hash(key, 0, 6) % np.uint64(3)).astype(np.int64), 0)
    for extra in range(3):
        m = trail > extra
        state[m, ncols[m] + extra] = 1
    ncols = ncols + trail
    cols = np.arange(cap)
    valid = cols[None, :] < ncols[:, None]
    consumes_q = valid & (state != 1)
    qi = np.cumsum(consumes_q, axis=1) - 1
    tt = np.broadcast_to(cols[None, :], (n, cap))
    qres = aa[(_hash(key[:, None], np.clip(qi, 0, None), 7) % np.uint64(20)).astype(np.int64)]      # residue qi of the query
    rnd = aa[(_hash(key[:, None], tt, 8) % np.uint64(20)).astype(np.int64)]
    keep = _u01(_hash(key[:, None], tt, 9)) < 0.6
    gq = np.where(state == 1, ord("-"), qres).astype(np.uint8)
    gt = np.where(state == 2, ord("-"), np.where((state == 0) & keep, qres, rnd)).astype(np.uint8)
    Lt = (valid & (state != 2)).sum(axis=1)
    gapped_q = [gq[i, :ncols[i]].tobytes().decode() for i in range(n)]
    gapped_t = [gt[i, :ncols[i]].tobytes().decode() for i in range(n)]
    seqs = [s.replace("-", "") for s in gapped_q]
    # ---- structures: random walk over the target residues, longest first so that every step only touches the live prefix
    order = np.argsort(-Lt, kind="stable")
    ko, Lo = key[order], Lt[order]
    Lmax = int(Lo[0]) if n else 0
    pos = np.zeros((n, 3))
    vprev = np.zeros((n, 3))
    out = np.zeros((Lmax, n, 3), np.float32)
    live = n
    for t in range(Lmax):
        while live > 0 and Lo[live - 1] <= t:
            live -= 1
        if t:
            kk = ko[:live]
            r1 = np.sqrt(-2.0 * np.log(_u01(_hash(kk, t, 10))))
            r2 = np.sqrt(-2.0 * np.log(_u01(_hash(kk, t, 11))))
            a1, a2 = 2.0 * np.pi * _u01(_hash(kk, t, 12)), 2.0 * np.pi * _u01(_hash(kk, t, 13))
            v = np.stack([r1 * np.cos(a1), r1 * np.sin(a1), r2 * np.cos(a2)], axis=1)
            v /= np.linalg.norm(v, axis=1, keepdims=True) + 1e-12
            v += 0.5 * vprev[:live]
            v /= np.linalg.norm(v, axis=1, keepdims=True) + 1e-12
            pos[:live] += 3.8 * v
            vprev[:live] = v
        out[t, :live] = np.round(pos[:live], 3)
    inv = np.empty(n, np.int64)
    inv[order] = np.arange(n)
    coords = [np.ascontiguousarray(out[:Lt[i], inv[i]]) for i in range(n)]
    return Workload(seqs, gapped_q, gapped_t, coords, threshold, generated_contacts, name or f"keyed_seed{seed}_n{n}")


def keyed_workload_parallel(ids: Sequence[int], seed: int, procs: int, block: int = 4096, **kw) -> Workload:
    """`keyed_workload` over a process pool (fork; call before CUDA is initialised in this process)."""
    ids = np.asarray(ids, np.int64)
    parts = [ids[i:i + block] for i in range(0, len(ids), block)]
    if procs <= 1 or len(parts) <= 1:
        ws = [keyed_workload(p, seed, **kw) for p in parts]
    else:
        import multiprocessing as mp
        from functools import partial
        with mp.get_context("fork").Pool(min(procs, len(parts))) as pool:
            ws = pool.map(partial(keyed_workload, seed=seed, **kw), parts)
    out = Workload([], [], [], [], kw.get("threshold", 10.0), kw.get("generated_contacts", 2), f"keyed_seed{seed}_n{len(ids)}")
    for w in ws:
        out.query_seqs += w.query_seqs
        out.gapped_query += w.gapped_query
        out.gapped_target += w.gapped_target
        out.coords += w.coords
    return out


ONE_TO_THREE = {"A": "ALA", "R": "ARG", "N": "ASN", "D": "ASP", "C": "CYS", "Q": "GLN", "E": "GLU", "G": "GLY", "H": "HIS", "I": "ILE",
                "L": "LEU", "K": "LYS", "M": "MET", "F": "PHE", "P": "PRO", "S": "SER", "T": "THR", "W": "TRP", "Y": "TYR", "V": "VAL"}


def pdb_text(seq: str, ca: np.ndarray, rng: Optional[np.random.Generator] = None, chain: str = "A", *, backbone: bool = True,
             extra_chain: bool = False, hetatm: bool = False, altloc_every: int = 0, models: int = 1, crlf: bool = False,
             first_res: int = 1) -> str:
    """A PDB file (fixed-column ATOM records, the text FoldComp decompresses to, `pdb.py:150-156`) holding `seq` with C-alpha
    atoms at `ca` [L, 3] - plus, optionally, what a parser has to skip: N / C / O backbone atoms, a second chain, HETATM records
    (a calcium ion named "CA", a modified residue), alternate locations, further models, CRLF line ends."""
    rng = rng or np.random.default_rng(0)
    lines: List[str] = ["HEADER    SYNTHETIC STRUCTURE", "CRYST1    1.000    1.000    1.000  90.00  90.00  90.00 P 1           1"]
    serial = [0]

    def atom(rec, name, alt, res, ch, num, xyz, elem):
        serial[0] += 1
        nm = f" {name:<3s}" if len(name) < 4 and len(elem) == 1 else f"{name:<4s}"
        lines.append(f"{rec:<6s}{serial[0] % 100000:5d} {nm}{alt}{res:>3s} {ch}{num:4d}    {xyz[0]:8.3f}{xyz[1]:8.3f}{xyz[2]:8.3f}{1.0:6.2f}{rng.uniform(20, 90):6.2f}"
                     f"          {elem:>2s}")

    def write_chain(ch, residues, cas, shift):
        for i, (r, c) in enumerate(zip(residues, cas)):
            res, num = ONE_TO_THREE[r], first_res + i
            c = np.asarray(c, np.float64) + shift
            alts = ["A", "B"] if altloc_every and i % altloc_every == altloc_every - 1 else [" "]
            if backbone:
                atom("ATOM", "N", " ", res, ch, num, c + [-1.2, 0.4, 0.3], "N")
            for k, alt in enumerate(alts):
                atom("ATOM", "CA", alt, res, ch, num, c + 0.25 * k, "C")
            if backbone:
                atom("ATOM", "C", " ", res, ch, num, c + [1.1, 0.7, -0.2], "C")
                atom("ATOM", "O", " ", res, ch, num, c + [1.6, 1.8, -0.4], "O")
        lines.append(f"TER   {serial[0] + 1:5d}      {ONE_TO_THREE[residues[-1]]:>3s} {ch}{first_res + len(residues) - 1:4d}" if residues else "TER")

    for m in range(models):
        if models > 1:
            lines.append(f"MODEL     {m + 1:4d}")
        if extra_chain and chain != "B":
            write_chain("B", seq[:max(1, len(seq) // 3)], ca[:max(1, len(seq) // 3)], np.array([50.0, 0.0, 0.0]))
        write_chain(chain, seq, ca, np.zeros(3) + 0.5 * m)
        if hetatm:
            atom("HETATM", "CA", " ", "CA", chain, first_res + len(seq) + 1, np.array([1.0, 2.0, 3.0]), "CA")      # a calcium ion
            atom("HETATM", "CA", " ", "MSE", chain, first_res + len(seq) + 2, np.array([4.0, 5.0, 6.0]), "C")       # modified residue
            atom("HETATM", "O", " ", "HOH", chain, first_res + len(seq) + 3, np.array([7.0, 8.0, 9.0]), "O")
        if models > 1:
            lines.append("ENDMDL")
    lines.append("END")
    return ("\r\n" if crlf else "\n").join(lines) + ("\r\n" if crlf else "\n")


def config_workload(idx: int, scale: float = 1.0) -> Workload:
    """BASELINE.json `configs[idx]`; `scale` shrinks the protein count for tests."""
    if idx == 0:
        return make_workload(max(1, int(1000 * scale)), 100, 500, seed=1, name="config0_1k_L100-500_MF")
    if idx == 1:
        return make_workload(max(1, int(100_000 * scale)), 50, 1000, seed=2, threshold=6.0,
                             name="config1_100k_pairs_cmap_transfer")
    if idx == 2:
        return make_workload(max(1, int(10_000 * scale)), 50, 1000, seed=3, dist="lognormal",
                             name="config2_10k_L50-1000_4heads")
    if idx == 3:
        return make_workload(max(1, int(2000 * scale)), 1000, 2500, seed=4, name="config3_2k_L1000-2500")
    if idx == 4:
        return make_workload(max(1, int(1_000_000 * scale)), 50, 1000, seed=5, dist="lognormal",
                             name="config4_1M_MF_sharded")
    raise ValueError(idx)
