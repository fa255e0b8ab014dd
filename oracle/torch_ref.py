"""ORACLE — TEST INFRASTRUCTURE ONLY (never imported by the product package).

Second, third-party-arithmetic executor of the DeepFRI `.onnx` files: the same graphs that
`oracle/gcn_oracle.py` interprets with hand-written NumPy formulas are executed here on PyTorch's CPU
kernels — `torch.nn.LSTM` (gate rows permuted from ONNX's i,o,f,c to torch's i,f,g,o), `F.conv1d` /
`F.conv2d`, `F.elu`, `F.batch_norm`, `torch.softmax`, `torch.matmul`.  PyTorch stands where the reference
has onnxruntime (`predict.pyx:62-73,98`; absent from this image): an independent implementation of the
published ONNX operator semantics (opset 15), decoded by `oracle/onnx_pb.py` (Google protobuf runtime).
`tests/test_oracle_torch.py` requires the NumPy oracle and this executor to agree to <= 1e-5 on every
golden case, so a shared misreading of the LSTM weight layout, the gate order, the bias split, the
Conv padding or the [C, 2] reshape would have to be made three times (here, in the NumPy oracle and in the
float64 layer-equation restatement of `oracle/gcn_f64.py`) to go unnoticed.
"""
from __future__ import annotations

import os
import sys
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn.functional as F

_HERE = os.path.dirname(os.path.abspath(__file__))
if _HERE not in sys.path:
    sys.path.insert(0, _HERE)
import onnx_pb  # noqa: E402

_ALPHABET = "-DGULNTKHYWCPVSOIEFXQABZRM"      # predict.pyx:26

_TORCH_OF = {1: torch.float32, 2: torch.uint8, 3: torch.int8, 6: torch.int32, 7: torch.int64, 9: torch.bool,
             10: torch.float16, 11: torch.float64}


def seq2onehot(seq: str) -> np.ndarray:
    """`predict.pyx:17-48` restated with torch's one_hot."""
    idx = []
    for ch in seq.encode("ascii").decode("ascii"):
        k = _ALPHABET.find(ch)
        if k < 0:
            raise ValueError(f"Invalid character in sequence: {ch}")
        idx.append(k)
    if not idx:
        return np.zeros((0, 26), np.float32)
    return F.one_hot(torch.tensor(idx), 26).to(torch.float32).numpy()


def _torch_lstm_module(W, R, B, H, dtype):
    """torch.nn.LSTM holding the weights of one ONNX LSTM node: W [1, 4H, I], R [1, 4H, H], B [1, 8H] = [Wb | Rb], ONNX gate
    order i, o, f, c.  torch stacks its rows as i, f, g(cell), o and keeps the two bias halves apart as bias_ih / bias_hh."""
    if W.shape[0] != 1:
        raise NotImplementedError("bidirectional LSTM")
    perm = torch.cat([torch.arange(0, H), torch.arange(2 * H, 3 * H), torch.arange(3 * H, 4 * H), torch.arange(H, 2 * H)])
    lstm = torch.nn.LSTM(input_size=W.shape[2], hidden_size=H, num_layers=1, bias=True, batch_first=False).to(dtype)
    with torch.no_grad():
        lstm.weight_ih_l0.copy_(W[0][perm])
        lstm.weight_hh_l0.copy_(R[0][perm])
        if B is not None:
            lstm.bias_ih_l0.copy_(B[0, :4 * H][perm])
            lstm.bias_hh_l0.copy_(B[0, 4 * H:][perm])
        else:
            lstm.bias_ih_l0.zero_()
            lstm.bias_hh_l0.zero_()
    return lstm


def _onnx_lstm(X, W, R, B, H, init_h, init_c, dtype, cache=None, key=None):
    """ONNX LSTM (forward, layout 0) on X [T, b, I] -> (Y [T, 1, b, H], Y_h, Y_c)."""
    lstm = cache.get(key) if cache is not None else None
    if lstm is None:
        lstm = _torch_lstm_module(W, R, B, H, dtype)
        if cache is not None:
            cache[key] = lstm
    with torch.no_grad():
        b = X.shape[1]
        h0 = torch.zeros(1, b, H, dtype=dtype) if init_h is None else init_h.to(dtype)
        c0 = torch.zeros(1, b, H, dtype=dtype) if init_c is None else init_c.to(dtype)
        Y, (hn, cn) = lstm(X, (h0, c0))
    return Y.unsqueeze(1), hn, cn          # ONNX Y is [T, num_directions, b, H]


def _pads(a, kshape):
    nsp = len(kshape)
    auto = a.get("auto_pad", "NOTSET")
    if auto in ("SAME_UPPER", "SAME_LOWER"):
        tot = [k - 1 for k in kshape]
        beg = [t // 2 if auto == "SAME_UPPER" else t - t // 2 for t in tot]
        return beg, [t - b for t, b in zip(tot, beg)]
    if auto == "VALID":
        return [0] * nsp, [0] * nsp
    p = [int(v) for v in a.get("pads", [0] * (2 * nsp))]
    return p[:nsp], p[nsp:]


class TorchOnnx:
    """Runs an ONNX inference graph on PyTorch CPU ops.  `dtype=torch.float64` runs every float tensor in double
    precision (used to tell fp32 round-off from a real disagreement)."""

    def __init__(self, model_path: str, dtype: torch.dtype = torch.float32):
        self.model = onnx_pb.load(model_path)
        self.graph = self.model.graph
        self.dtype = dtype
        self.input_names = [v.name for v in self.graph.inputs]
        self.output_names = [v.name for v in self.graph.outputs]
        self.const = {k: self._t(v) for k, v in self.graph.initializers.items()}
        self._lstm_modules = {}       # one torch.nn.LSTM per LSTM node, built on first use (constant weights)

    def _t(self, a) -> torch.Tensor:
        t = torch.from_numpy(np.array(a, copy=True)) if isinstance(a, np.ndarray) else torch.as_tensor(a)
        return t.to(self.dtype) if t.is_floating_point() else t

    def _node(self, n, v: Dict[str, torch.Tensor]) -> List[torch.Tensor]:
        def inp(k):
            return v[n.inputs[k]] if k < len(n.inputs) and n.inputs[k] != "" else None

        def axes_of(k):
            ax = inp(k) if inp(k) is not None else n.attrs.get("axes")
            return None if ax is None else [int(x) for x in torch.as_tensor(ax).reshape(-1).tolist()]
        a, op = n.attrs, n.op_type
        if op == "MatMul":
            return [torch.matmul(inp(0), inp(1))]
        if op == "Gemm":
            A = inp(0).T if a.get("transA", 0) else inp(0)
            Bm = inp(1).T if a.get("transB", 0) else inp(1)
            y = float(a.get("alpha", 1.0)) * (A @ Bm)
            return [y + float(a.get("beta", 1.0)) * inp(2) if inp(2) is not None else y]
        if op in ("Add", "Sub", "Mul", "Div"):
            return [{"Add": torch.add, "Sub": torch.sub, "Mul": torch.mul, "Div": torch.div}[op](inp(0), inp(1))]
        if op == "Sqrt":
            return [torch.sqrt(inp(0))]
        if op == "Reciprocal":
            return [torch.reciprocal(inp(0))]
        if op == "Relu":
            return [F.relu(inp(0))]
        if op == "Elu":
            return [F.elu(inp(0), alpha=float(a.get("alpha", 1.0)))]
        if op == "Sigmoid":
            return [torch.sigmoid(inp(0))]
        if op == "Tanh":
            return [torch.tanh(inp(0))]
        if op == "Softmax":
            return [torch.softmax(inp(0), dim=int(a.get("axis", -1)))]
        if op == "Transpose":
            return [inp(0).permute(*a["perm"])]
        if op == "Squeeze":
            ax = axes_of(1)
            x = inp(0)
            if ax is None:
                return [x.squeeze()]
            for d in sorted((d % x.dim() for d in ax), reverse=True):
                x = x.squeeze(d)
            return [x]
        if op == "Unsqueeze":
            x = inp(0)
            for d in sorted(axes_of(1)):
                x = x.unsqueeze(d)
            return [x]
        if op == "Reshape":
            x, shp = inp(0), [int(s) for s in inp(1).tolist()]
            return [x.reshape([x.shape[i] if s == 0 else s for i, s in enumerate(shp)])]
        if op == "Concat":
            return [torch.cat([v[i] for i in n.inputs], dim=int(a["axis"]))]
        if op == "ReduceSum":
            ax = axes_of(1)
            keep = bool(a.get("keepdims", 1))
            return [inp(0).sum() if ax is None else inp(0).sum(dim=ax, keepdim=keep)]
        if op == "ReduceMax":
            ax = axes_of(1)
            return [torch.amax(inp(0), dim=ax, keepdim=bool(a.get("keepdims", 1)))]
        if op == "GlobalMaxPool":
            x = inp(0)
            return [torch.amax(x, dim=list(range(2, x.dim())), keepdim=True)]
        if op == "EyeLike":
            x = inp(0)
            if a.get("k", 0) != 0:
                raise NotImplementedError("EyeLike k != 0")
            return [torch.eye(x.shape[0], x.shape[1], dtype=x.dtype)]
        if op == "Shape":
            return [torch.tensor(list(inp(0).shape), dtype=torch.int64)]
        if op == "Gather":
            return [torch.index_select(inp(0), int(a.get("axis", 0)), inp(1).reshape(-1)).reshape(
                list(inp(0).shape[:int(a.get("axis", 0))]) + list(inp(1).shape) + list(inp(0).shape[int(a.get("axis", 0)) + 1:]))]
        if op == "Cast":
            to = _TORCH_OF[a["to"]]
            return [inp(0).to(self.dtype if to.is_floating_point else to)]
        if op in ("Identity", "Dropout"):
            return [inp(0)]
        if op == "Constant":
            return [self._t(a["value"])]
        if op == "Slice":
            x = inp(0)
            starts, ends = inp(1).tolist(), inp(2).tolist()
            axes = inp(3).tolist() if inp(3) is not None else list(range(len(starts)))
            steps = inp(4).tolist() if inp(4) is not None else [1] * len(starts)
            sl = [slice(None)] * x.dim()
            for s, e, ax, st in zip(starts, ends, axes, steps):
                sl[int(ax)] = slice(int(s), int(e), int(st))
            return [x[tuple(sl)]]
        if op == "Conv":
            x, w, b = inp(0), inp(1), inp(2)
            if a.get("group", 1) != 1:
                raise NotImplementedError("grouped Conv")
            kshape = list(w.shape[2:])
            beg, end = _pads(a, kshape)
            pad = []
            for bb, ee in reversed(list(zip(beg, end))):      # F.pad counts from the last axis
                pad += [bb, ee]
            x = F.pad(x, pad)
            strides = [int(s) for s in a.get("strides", [1] * len(kshape))]
            dil = [int(s) for s in a.get("dilations", [1] * len(kshape))]
            conv = {1: F.conv1d, 2: F.conv2d}[len(kshape)]
            return [conv(x, w, b, stride=strides, dilation=dil)]
        if op == "BatchNormalization":
            x, sc, bi, mean, var = (inp(k) for k in range(5))
            return [F.batch_norm(x, mean, var, sc, bi, training=False, eps=float(a.get("epsilon", 1e-5)))]
        if op == "LSTM":
            if a.get("direction", "forward") != "forward" or a.get("layout", 0) != 0:
                raise NotImplementedError("LSTM: only forward / layout 0")
            if "activations" in a and [s.lower() for s in a["activations"]] != ["sigmoid", "tanh", "tanh"]:
                raise NotImplementedError("LSTM with non-default activations")
            if inp(7) is not None:
                raise NotImplementedError("LSTM peepholes")
            X = inp(0)
            if inp(4) is not None and any(int(s) != X.shape[0] for s in inp(4).reshape(-1).tolist()):
                raise NotImplementedError("LSTM sequence_lens shorter than the sequence")
            const_w = all(k in self.const for k in n.inputs[1:4] if k)
            return list(_onnx_lstm(X, inp(1), inp(2), inp(3), int(a["hidden_size"]), inp(5), inp(6), self.dtype,
                                   self._lstm_modules if const_w else None, n.outputs[0]))
        raise NotImplementedError(f"torch_ref: ONNX op {op} not implemented")

    def run(self, output_names: Optional[List[str]], feeds: Dict[str, np.ndarray]) -> List[np.ndarray]:
        v = dict(self.const)
        for k, x in feeds.items():
            v[k] = self._t(np.asarray(x))
        with torch.no_grad():
            for n in self.graph.nodes:
                for name, val in zip(n.outputs, self._node(n, v)):
                    if name:
                        v[name] = val
        return [v[k].numpy() for k in (output_names or self.output_names)]


class Predictor:
    """Twin of `mDeepFRI.predict.Predictor` (`predict.pyx:50-102`) over `TorchOnnx`."""

    def __init__(self, model_path: str, threads: int = 1, dtype: torch.dtype = torch.float32):
        self.model_path, self.threads = model_path, threads
        self.session = TorchOnnx(model_path, dtype)
        self.input_names = self.session.input_names

    def forward_pass(self, seqres: str, cmap=None) -> np.ndarray:
        S = seq2onehot(seqres)
        S = S.reshape(1, *S.shape)
        if cmap is None:
            feeds = {self.input_names[0]: S}
        else:
            A = np.asarray(cmap).reshape(1, cmap.shape[0], cmap.shape[1]).astype(np.float32)
            feeds = {self.input_names[0]: A, self.input_names[1]: S}
        y = self.session.run(None, feeds)[0]
        return y[:, :, 0].reshape(-1).astype(np.float32)
